#!/usr/bin/env python
"""bench.py -- SIPP native prover benchmark (BASELINE.json metric: pairings aggregated per second at n = 2^k).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--n PAIRS] [--impl reference] [--dump-outputs DIR]

A "step" is one complete `sipp_prove_native` of n random BN254 pairs (seeded synthetic inputs): Z, then log2(n)
rounds of (Z_L, Z_R multi-pairings, Poseidon challenge, G1/G2 folds).  N = 1 runs BASELINE configs[1]
(n = 2^12, one B200); N > 1 runs the strided-shard multi-GPU prover with 2^12 pairs per GPU (weak scaling).

  value  pairs/s with the inputs already resident in HBM (the host still runs the transcript, which needs the
         host copy of A, B -- it is part of the job)
  e2e    pairs/s through the public call `sipp_prove_native(A, B)` with HOST buffers: H2D of A, B and D2H of every
         Z / the proof inside the timed region
  roofline   Miller-loop kernel: algorithmic IMAD-pipe instructions (9,008 Fq-mul x 264 per pair, SURVEY 8d) / its
         CUDA-event time in the timed region, against the measured IMAD peak (microbenchmark in the same run)
  cpu_baseline  the oracle (CPU restatement of the reference) on a bounded sample, timed on this box's host cores

`--impl reference` times the CPU restatement of the reference prover (oracle/, faithful structure: one full
pairing per pair) with all host threads on the same config.

`--dump-outputs DIR` writes the proofs of the last timed step as DIR/<name>.npy, so that two builds can be compared
output for output (the inputs are seeded: the same arguments give the same inputs).  Each proof element is an Fq12 of
12 coefficients of 8 little-endian u32 limbs, stored as float64 limb values (exact):
  proof.npy                  [2 log2(n) + 1, 12, 8]  the headline proof (seed 2; `--impl reference`: of the pairs it times)
  proof_n2p16.npy, ...       the BASELINE large configurations of the default line, when they run
  batch_proofs.npy           [instances, 2 log2(n) + 1, 12, 8]  batched instances (--workload batch, or the default
  batch_instances.npy        line's config-5 step) and their instance indices; beyond 64 MB in all, a fixed seeded
                             sample of the instances
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FQMUL_PER_MILLER = 9008      # SURVEY 8(d) / Appendix C: 64 x 107 + 27 x 80
IMAD_PER_FQMUL = 264         # 8x32-bit CIOS Montgomery: 128 product halves + 136 reduction
PAIRS_PER_GPU = 1 << 12
# DRAM bytes per launch of the dominant kernels (dram__bytes_read.sum + dram__bytes_write.sum) from the ncu --set full captures
# under profiles/ (tools/ncu_traffic.sh writes them); None until a capture of the current kernels is committed
NCU_TRAFFIC = {}
try:
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")) as _f:
        NCU_TRAFFIC = json.load(_f)
except Exception:
    pass


def log2(n):
    return n.bit_length() - 1


def miller_loops_per_prove(n):
    return 3 * n - 2


class ClockSampler:
    """samples the SM clock and the throttle reasons during the timed region (B200_PROFILING.md recipe: the clocks line of
    nvidia-smi).  Read through NVML in-process -- the same counters `nvidia-smi --query-gpu=clocks.sm,clocks.max.sm,
    clocks_event_reasons.*` prints -- because forking nvidia-smi five times a second from this process stole the core of the host
    thread that runs the transcript chain (a resident step measured 69 ms with it, 52.5 ms without); nvidia-smi itself is the
    fallback when the NVML binding is missing."""

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], False
        self.t = threading.Thread(target=self._run, daemon=True)
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = (pynvml, pynvml.nvmlDeviceGetHandleByIndex(index))
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        nv, h = self.nvml
        sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        r = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        bits = [("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4)]
        return [str(sm), str(mx), "0"] + ["Active" if r & b else "Not Active" for _, b in bits]

    def _run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop:
            try:
                if self.nvml:
                    self.rows.append(self._sample_nvml())
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.05 if self.nvml else 0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "NVML (pynvml)" if self.nvml else "nvidia-smi"}


def run_reference(args):
    """the reference arm: CPU restatement of prover_native.rs (oracle), all host threads, rank 0 only"""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import pyoracle as o
    cores = os.cpu_count() or 1
    if args.workload == "batch":
        # config 5 on the host cores: instances are independent, so a step proves ONE instance with every core working on it
        # (the oracle parallelises the pairings of a product); work per instance is identical, instances/s = 1 / step
        n = args.instance_n
        A, B = o.seeded_inputs(5, n, threads=cores)
        for _ in range(args.warmup):
            o.sipp_prove(A[:64 * 32], B[:128 * 32], o.FAITHFUL, cores)
        times = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            proof = o.sipp_prove(A, B, o.FAITHFUL, cores)
            times.append(time.perf_counter() - t0)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {}, (proof, len(proof) // 384, 0))
        per_step = sum(times) / len(times)
        value = 1.0 / per_step
        print(json.dumps({"impl": "reference", "metric": "SIPP native prove throughput, batched independent instances (instances per second)",
                          "value": value, "unit": "instances/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                          "dtype": "u32 limbs (254-bit modular integer)", "data": "synthetic",
                          "config": {"workload": "batched throughput: %d independent n=%d SIPP instances (CPU restatement of the reference)"
                                                 % (args.instances, n), "instances": args.instances, "n": n},
                          "cpu_baseline": {"value": value, "unit": "instances/s", "cores": cores, "kind": "port",
                                           "sample": "one faithful n=%d prove per step with all %d host threads; the %d instances are identical "
                                                     "work" % (n, cores, args.instances)},
                          "e2e": {"value": value, "unit": "instances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0
    n = args.n or PAIRS_PER_GPU * args.gpus
    A, B = o.seeded_inputs(2, n, threads=cores)
    # one step = one faithful prove of the whole configuration (n = 2^12: ~1.4 s with 16 threads); beyond 2^15 pairs a step is
    # the first 2^15 pairs (work is linear in n) so that the run stays within minutes
    sample_n = min(n, 1 << 15)
    As, Bs = A[:64 * sample_n], B[:128 * sample_n]
    for _ in range(args.warmup):
        o.sipp_prove(As[:64 * 32], Bs[:128 * 32], o.FAITHFUL, cores)
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        proof = o.sipp_prove(As, Bs, o.FAITHFUL, cores)
        times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"proof": proof})
    per_step = sum(times) / len(times)
    value = sample_n / per_step
    t0 = time.perf_counter()
    o.sipp_prove(As[:64 * 128], Bs[:128 * 128], o.FAITHFUL, 1)   # the reference as written is single-threaded
    single = 128 / (time.perf_counter() - t0)
    line = {"impl": "reference", "metric": "SIPP native prove throughput (pairings aggregated per second)", "value": value,
            "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (254-bit modular integer)",
            "data": "synthetic", "config": {"workload": "SIPP native prover, n=%d pairs (CPU restatement of the reference; "
                                                        "no Rust toolchain, see DESIGN.md)" % n, "n": n},
            "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": "port",
                             "sample": ("faithful prove (one full pairing per pair, naive folds, Poseidon transcript) of all %d pairs per step" % n)
                             if sample_n == n else ("faithful prove of the first %d of %d pairs per step; work is linear in n" % (sample_n, n)),
                             "same_config": sample_n == n,
                             "single_thread": {"value": single, "unit": "pairs/s", "cores": 1,
                                               "sample": "faithful prove of 128 pairs on one thread (the reference itself is single-threaded)"}},
            "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def measure_batch(count_total, n, world, rank, local_rank, W, K, barrier, all_max, flush):
    """BASELINE config 5: `count_total` independent n-pair instances proved in lock-step, each with its own Fiat-Shamir chain on
    the device; rank g owns a contiguous slice of the instances (no collective).  Returns a dict of measurements."""
    import ctypes
    import torch
    import sipp_b200
    from sipp_b200 import _lib
    from sipp_b200.sharded import shard_instances
    lib = _lib.load()
    lo, hi = shard_instances(count_total, rank, world)
    count = hi - lo
    plen = lib.sipp_proof_len(n)
    total = n * count
    # instance j is seeded_inputs(seed = 5)[j * n : (j + 1) * n]: generate the global stream, keep this rank's slice
    gA = torch.empty(count_total * n * 64, dtype=torch.uint8, device="cuda")
    gB = torch.empty(count_total * n * 128, dtype=torch.uint8, device="cuda")
    _lib.check(lib.sipp_seeded_inputs_device(5, count_total * n, gA.data_ptr(), gB.data_ptr()))
    dA = gA[lo * n * 64:hi * n * 64].clone()
    dB = gB[lo * n * 128:hi * n * 128].clone()
    del gA, gB
    dP = torch.empty(count * plen * 384, dtype=torch.uint8, device="cuda")
    A_pin, B_pin = dA.cpu().pin_memory(), dB.cpu().pin_memory()
    P_pin = torch.empty(count * plen * 384, dtype=torch.uint8).pin_memory()

    def step_resident():
        _lib.check(lib.sipp_prove_native_batch_device(dA.data_ptr(), dB.data_ptr(), n, count, dP.data_ptr()))

    def step_e2e():
        _lib.check(lib.sipp_prove_native_batch(ctypes.c_char_p(A_pin.data_ptr()), ctypes.c_char_p(B_pin.data_ptr()), n, count,
                                               ctypes.c_char_p(P_pin.data_ptr())))

    def timed(fn, steps):
        tot = 0.0
        for _ in range(steps):
            flush()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            t0 = time.perf_counter()
            fn()
            e1.record()
            barrier()
            tot += all_max(max(time.perf_counter() - t0, e0.elapsed_time(e1) * 1e-3))
        return tot

    for _ in range(W):
        step_resident()
    sipp_b200.stats(reset=True)
    t_res = timed(step_resident, K)
    launches = sipp_b200.stats(reset=True)["launches"]
    # kernel-class shares and the roofline come from a separate profiled pass: with event spans on, the library runs the batch as
    # one sub-batch so that the spans do not overlap (the timed steps above overlap sub-batches on several streams)
    sipp_b200.set_option(_lib.OPT_PROFILE, 1)
    sipp_b200.stats(reset=True)
    t_prof = timed(step_resident, 1)
    st = sipp_b200.stats(reset=True)
    sipp_b200.set_option(_lib.OPT_PROFILE, 0)
    st["launches"] = launches
    st["profiled_step_ms"] = t_prof * 1e3
    for _ in range(W):
        step_e2e()
    t_e2e = timed(step_e2e, K)
    proofs = dP.cpu().numpy().tobytes()
    assert proofs == P_pin.numpy().tobytes(), "resident and e2e batch proofs differ"
    # parity inside the run: a sample of this rank's instances against the single-instance prover (itself pinned to the oracle)
    A, B = A_pin.numpy().tobytes(), B_pin.numpy().tobytes()
    for j in sorted({0, count // 2, count - 1}):
        a, b = A[64 * n * j:64 * n * (j + 1)], B[128 * n * j:128 * n * (j + 1)]
        assert proofs[j * plen * 384:(j + 1) * plen * 384] == b"".join(sipp_b200.sipp_prove_native(a, b)), "batch instance %d differs" % j
    return {"count": count, "t_res": t_res, "t_e2e": t_e2e, "stats": st, "h2d": total * 192, "d2h": count * plen * 384,
            "sample": (A[:64 * n], B[:128 * n], proofs[:plen * 384]), "proofs": (proofs, plen, lo)}


def run_batch(args, world, rank, local_rank, W, K):
    import ctypes
    import torch
    import torch.distributed as dist
    import sipp_b200
    from sipp_b200 import _lib
    lib = _lib.load()
    n, count_total = args.instance_n, args.instances
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def flush():
        flush_buf.zero_()
        torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_max(dt):
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return dt

    with ClockSampler(local_rank) as clocks:
        m = measure_batch(count_total, n, world, rank, local_rank, W, K, barrier, all_max, flush)
    clk = clocks.summary()
    peaks = {}
    for which, name in ((0, "mad_lo"), (1, "mad_wide"), (2, "mad_lo_hi_carry"), (3, "fq_mul_ptx")):
        ops, ms = ctypes.c_double(), ctypes.c_double()
        _lib.check(lib.sipp_microbench(which, 2000 if which < 3 else 400, ctypes.byref(ops), ctypes.byref(ms)))
        peaks[name] = ops.value
    imad_peak = max(peaks["mad_lo"], 2 * peaks["mad_wide"], peaks["mad_lo_hi_carry"])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {}, m["proofs"])
    st = m["stats"]
    mill_ach = st["miller_pairs"] * FQMUL_PER_MILLER * IMAD_PER_FQMUL / max(st["miller_ms"] * 1e-3, 1e-12)
    line = {"metric": "SIPP native prove throughput, batched independent instances (instances per second)", "value": count_total * K / m["t_res"],
            "unit": "instances/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": m["t_res"] / K * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u32 limbs (254-bit modular integer)", "data": "synthetic",
            "config": {"workload": "batched throughput: %d independent n=%d SIPP instances, %dxB200 (instances sharded by rank, no collective)"
                                   % (count_total, n, world), "instances": count_total, "n": n, "seed": 5,
                       "miller_loops_per_step": count_total * miller_loops_per_prove(n), "l2": "flushed between steps (256 MB write)",
                       "transcript": "on the device, one Poseidon chain per instance"},
            "pairs_per_s": count_total * n * K / m["t_res"],
            "e2e": {"value": count_total * K / m["t_e2e"], "unit": "instances/s", "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": m["d2h"],
                    "ms_per_step": m["t_e2e"] / K * 1e3},
            "gpu_launches": int(st["launches"]), "clocks": clk,
            "roofline": {"bound": "imad", "kernel": "k_lines_batch + k_accum (Miller loops of all instances of a round)", "achieved": mill_ach / 1e12,
                         "peak": imad_peak / 1e12, "unit": "T IMAD/s", "frac": mill_ach / imad_peak, "traffic": None,
                         "launches": int(st["miller_launches"]), "avg_launch_ms": st["miller_ms"] / max(1, st["miller_launches"]),
                         "peak_source": "measured in this run (sipp_microbench); kernel times from one profiled step",
                         "kernel_time_share": {"miller_ms": st["miller_ms"], "final_exp_ms": st["reduce_fe_ms"], "fold_ms": st["fold_ms"],
                                               "decode_transcript_ms(side stream, overlapped)": st["other_ms"],
                                               "profiled_step_ms(single stream, event spans on)": st["profiled_step_ms"],
                                               "step_ms": m["t_res"] / K * 1e3},
                         "microbench": peaks}}
    if not args.no_cpu_baseline:
        from oracle import pyoracle as o
        a, b, gpu = m["sample"]
        cores = os.cpu_count() or 1
        t0 = time.perf_counter()
        ref = o.sipp_prove(a, b, o.FAITHFUL, 1)
        dt = time.perf_counter() - t0
        assert ref == gpu, "batch instance 0 differs from the oracle"
        line["cpu_baseline"] = {"value": 1.0 / dt, "unit": "instances/s", "cores": 1, "kind": "port",
                                "sample": "single-thread faithful restatement proving instance 0 (n=%d), %.2f s; byte-identical to the GPU's "
                                          "proof of that instance; %d host cores would run %d such instances side by side" % (n, dt, cores, cores)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def golden_large():
    """oracle digests of the BASELINE configurations (tests/golden/gen_large_digests.py wrote them; committed)"""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "sipp_large.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def measure_large(k, seed, world, rank, local_rank, barrier, all_max, flush):
    """One BASELINE large configuration (configs[2]: n = 2^16, configs[3]: n = 2^20) through the PUBLIC call with HOST buffers:
    every rank uploads its strided shard inside the timed region, rank 0 runs the transcript.  One timed prove (plus one
    warm-up for n <= 2^16), CUDA-event spans on.  The proof is compared with the oracle's digest of the same seeded inputs."""
    import hashlib
    import torch
    import sipp_b200
    from sipp_b200 import _lib
    from sipp_b200.sharded import sharded_prove
    lib = _lib.load()
    n = 1 << k
    dA = torch.empty(n * 64, dtype=torch.uint8, device="cuda")
    dB = torch.empty(n * 128, dtype=torch.uint8, device="cuda")
    t0 = time.perf_counter()
    _lib.check(lib.sipp_seeded_inputs_device(seed, n, dA.data_ptr(), dB.data_ptr()))   # fixed-base keygen on the GPU (k_seeded_inputs)
    t_gen = time.perf_counter() - t0
    Al = dA.view(n, 64)[rank::world].contiguous().cpu().pin_memory()
    Bl = dB.view(n, 128)[rank::world].contiguous().cpu().pin_memory()
    A = B = None
    if rank == 0:
        A, B = dA.cpu().numpy().tobytes(), dB.cpu().numpy().tobytes()
    del dA, dB
    torch.cuda.empty_cache()
    Alb, Blb = ctypes_ptr(Al), ctypes_ptr(Bl)

    def step():
        return sharded_prove(Alb, Blb, n, A, B)

    if k <= 16:
        step()
    sipp_b200.set_option(_lib.OPT_PROFILE, 1)
    sipp_b200.stats(reset=True)
    flush()
    barrier()
    t0 = time.perf_counter()
    proof = step()
    barrier()
    dt = all_max(time.perf_counter() - t0)
    st = sipp_b200.stats(reset=True)
    sipp_b200.set_option(_lib.OPT_PROFILE, 0)
    if rank != 0:
        return None
    g = golden_large().get("n=2^%d" % k)
    digest = hashlib.sha256(b"".join(proof)).hexdigest()
    ok = None
    if g is not None:
        assert hashlib.sha256(A).hexdigest() == g["sha256_A"] and hashlib.sha256(B).hexdigest() == g["sha256_B"], "seeded inputs differ from the oracle's"
        ok = digest == g["sha256_proof"]
        assert ok, "n = 2^%d proof differs from the oracle digest" % k
    return {"n": n, "seed": seed, "n_gpus": world, "prove_s": dt, "pairs_per_s": n / dt, "timed": "one prove through host buffers (H2D of every "
            "rank's shard and D2H of the proof inside), after %s" % ("one warm-up prove" if k <= 16 else "the n = 2^16 run as warm-up"),
            "h2d_bytes": n * 192, "d2h_bytes": 384 * (2 * k + 1), "sha256_proof": digest, "proof": b"".join(proof),
            "parity": ("bit-exact: sha256(proof) equals the oracle's digest (tests/golden/sipp_large.json)" if ok else "no golden digest for this size"),
            "rank0_kernel_ms": {"miller": st["miller_ms"], "reduce_final_exp": st["reduce_fe_ms"], "fold": st["fold_ms"], "other": st["other_ms"]},
            "host_transcript_exposed_ms": st["transcript_ms"], "miller_pairs_rank0": int(st["miller_pairs"]),
            "miller_loops_per_s_rank0": st["miller_pairs"] / max(st["miller_ms"] * 1e-3, 1e-12),
            "input_generation_s": t_gen}


def ctypes_ptr(t):
    import ctypes
    return ctypes.cast(t.data_ptr(), ctypes.c_char_p)


DUMP_BYTES_MAX = 64 << 20


def fq12_limbs(raw, plen):
    """proof bytes (384-byte Fq12 elements, plen per proof) -> float64 [proofs, plen, 12, 8] of the u32 limbs (all < 2^32: exact)"""
    import numpy as np
    return np.frombuffer(raw, dtype="<u4").astype(np.float64).reshape(-1, plen, 12, 8)


def dump_outputs(directory, proofs, batch=None):
    """--dump-outputs: `proofs` maps names to single proofs (bytes); `batch` = (bytes of consecutive proofs, elements per proof,
    index of the first instance).  The batch gets what the single proofs leave of the budget, as a fixed seeded sample of
    its instances if it does not fit."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    used = 0
    for name, raw in proofs.items():
        a = fq12_limbs(raw, len(raw) // 384)[0]
        np.save(os.path.join(directory, name + ".npy"), a)
        used += a.nbytes
    if batch is not None:
        raw, plen, first = batch
        a = fq12_limbs(raw, plen)
        keep = (DUMP_BYTES_MAX - used - 4096) // (a[0].nbytes + 8)    # 8 bytes for the index; 4096 for the .npy headers
        idx = np.arange(len(a)) if keep >= len(a) else np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))
        np.save(os.path.join(directory, "batch_proofs.npy"), a[idx])
        np.save(os.path.join(directory, "batch_instances.npy"), (idx + first).astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--n", "--pairs", dest="n", type=int, default=0, help="total pairs (default 2^12 per GPU); under torchrun spell it --pairs")
    ap.add_argument("--quick", action="store_true", help="large-n runs (n = 2^20): one warm-up step, no separate e2e leg (reported as null)")
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--saturated-pairs", type=int, default=1 << 17)
    ap.add_argument("--workload", default="prove", choices=["prove", "batch"],
                    help="prove: one n-pair proof (BASELINE configs[1], the default); batch: BASELINE config 5, independent "
                         "n=128 instances in lock-step, sharded by instance over the GPUs")
    ap.add_argument("--instances", type=int, default=4096)
    ap.add_argument("--instance-n", type=int, default=128)
    ap.add_argument("--batch-instances", type=int, default=4096, help="config-5 summary added to the default line (0 = skip)")
    ap.add_argument("--large", default="16,20", help="log2 sizes of the BASELINE large configurations added to the default line ('' = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the proofs of the last timed step to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import ctypes
    import torch
    import torch.distributed as dist
    import sipp_b200
    from sipp_b200 import _lib
    from sipp_b200.sharded import comm_init_torch, sharded_prove

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    os.environ["SIPP_DEVICE"] = str(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n = args.n or PAIRS_PER_GPU * world
    lib = _lib.load()
    _lib.require_gpu_once()
    if world > 1:
        comm_init_torch()   # NCCL communicator INSIDE the library (sipp_comm_init); torch only ships the 128-byte unique id
    W, K = (1 if args.quick else max(args.warmup, 3)), args.steps
    if args.workload == "batch":
        return run_batch(args, world, rank, local_rank, W, K)

    # ---- synthetic inputs (seeded, generated on the GPU; same stream as the oracle's generator) ----
    dA = torch.empty(n * 64, dtype=torch.uint8, device="cuda")
    dB = torch.empty(n * 128, dtype=torch.uint8, device="cuda")
    _lib.check(lib.sipp_seeded_inputs_device(2, n, dA.data_ptr(), dB.data_ptr()))
    A, B = dA.cpu().numpy().tobytes(), dB.cpu().numpy().tobytes()   # every rank: the single-GPU check below runs on rank 0 only
    dAl = dA.view(n, 64)[rank::world].contiguous()                   # strided ownership: rank g holds the pairs i = g (mod world)
    dBl = dB.view(n, 128)[rank::world].contiguous()
    Al_pin, Bl_pin = dAl.cpu().pin_memory(), dBl.cpu().pin_memory()
    del dA, dB
    A0, B0 = (A, B) if rank == 0 else (None, None)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def l2_flush():
        flush.zero_()
        torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_max(dt):
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return dt

    def timed(fn, steps):
        """K steps, each bracketed by barrier + synchronize; L2 flushed between steps outside the timed spans.
        Returns (seconds summed over steps as max over ranks, last result)."""
        total = 0.0
        res = None
        for _ in range(steps):
            l2_flush()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            t0 = time.perf_counter()
            res = fn()
            e1.record()
            barrier()
            total += all_max(max(time.perf_counter() - t0, e0.elapsed_time(e1) * 1e-3))
        return total, res

    # one code path for every N: the library's sharded prover (a world of one is sipp_prove_native on one GPU)
    def step_resident():
        return sharded_prove(None, None, n, A0, B0, device_ptrs=(dAl.data_ptr(), dBl.data_ptr()))

    def step_e2e():
        # the public call: host buffers in (pinned), proof out -- H2D of every rank's shard and D2H of the results inside
        return sharded_prove(ctypes_ptr(Al_pin), ctypes_ptr(Bl_pin), n, A0, B0)
    h2d = n * 192                       # summed over the ranks (each uploads its n / world pairs)
    d2h = 384 * (2 * log2(n) + 1)       # rank 0 reads every Z / Z_L / Z_R = the proof

    # ---- warm-up, then the timed region (profile spans on: CUDA events around every kernel class) ----
    for _ in range(W):
        step_resident()
    sipp_b200.set_option(_lib.OPT_PROFILE, 1)
    sipp_b200.stats(reset=True)
    with ClockSampler(local_rank) as clocks:
        t_res, proof_res = timed(step_resident, K)
        st = sipp_b200.stats(reset=True)
        sipp_b200.set_option(_lib.OPT_PROFILE, 0)
        if args.quick:
            t_e2e, proof_e2e = float("nan"), proof_res
        else:
            for _ in range(W):
                step_e2e()
            t_e2e, proof_e2e = timed(step_e2e, K)
    clk = clocks.summary()

    # ---- IMAD peak (microbenchmark, this GPU, this run) and the saturated Miller-kernel leg ----
    peaks = {}
    for which, name in ((0, "mad_lo"), (1, "mad_wide"), (2, "mad_lo_hi_carry"), (3, "fq_mul_ptx"), (4, "fq_mul_portable")):
        ops, ms = ctypes.c_double(), ctypes.c_double()
        _lib.check(lib.sipp_microbench(which, 2000 if which < 3 else 400, ctypes.byref(ops), ctypes.byref(ms)))
        peaks[name] = ops.value
    # peak of the integer-multiply pipe in 32x32 product-halves per second: a 32-bit IMAD retires one half, an
    # IMAD.WIDE (with or without carry) retires two but issues at half the rate, so all three legs agree (18.5 T/s)
    imad_peak = max(peaks["mad_lo"], 2 * peaks["mad_wide"], peaks["mad_lo_hi_carry"])
    sat = None
    if rank == 0 and args.saturated_pairs:
        m = args.saturated_pairs
        sA, sB = sipp_b200.seeded_inputs(3, 4096)
        reps = m // 4096
        ctx = sipp_b200.ProverContext(sA * reps, sB * reps)
        ctx.inner_product()
        sipp_b200.set_option(_lib.OPT_PROFILE, 1)
        sipp_b200.stats(reset=True)
        ctx.inner_product()
        s2 = sipp_b200.stats(reset=True)
        sipp_b200.set_option(_lib.OPT_PROFILE, 0)
        ctx.close()
        ach = s2["miller_pairs"] * FQMUL_PER_MILLER * IMAD_PER_FQMUL / (s2["miller_ms"] * 1e-3)
        sat = {"pairs": int(s2["miller_pairs"]), "miller_ms": s2["miller_ms"], "miller_loops_per_s": s2["miller_pairs"] / (s2["miller_ms"] * 1e-3),
               "kernels": "k_lines + k_accum", "achieved": ach / 1e12, "peak": imad_peak / 1e12, "unit": "T IMAD/s", "frac": ach / imad_peak,
               "algorithmic_input_bytes": m * 192,
               "traffic": {k: v.get("dram_bytes_per_launch") for k, v in ((NCU_TRAFFIC.get("saturated") or {}).get("kernels") or {}).items()} or None,
               "line_table_bytes": m * 29120}

    # ---- the other BASELINE configurations beside the headline (every rank takes part) ----
    large = []
    large_proofs = {}
    if not args.quick and not args.n:
        for k in [int(x) for x in args.large.split(",") if x]:
            r = measure_large(k, {16: 3, 20: 4}.get(k, 7), world, rank, local_rank, barrier, all_max, l2_flush)
            if r is not None:
                large_proofs["proof_n2p%d" % k] = r.pop("proof")
                r["miller_frac_of_imad_peak_rank0"] = r["miller_loops_per_s_rank0"] * FQMUL_PER_MILLER * IMAD_PER_FQMUL / imad_peak
                large.append(r)
    bm = None
    if args.batch_instances and not args.quick and not args.n:
        # BASELINE config 5 beside the headline (one timed step; `--workload batch` is the full bench of that config)
        bm = measure_batch(args.batch_instances, 128, world, rank, local_rank, 1, 1, barrier, all_max, l2_flush)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    import hashlib
    assert b"".join(proof_res) == b"".join(proof_e2e), "resident and e2e proofs differ"
    parity = None
    g = golden_large().get("seed2_n=2^%d" % log2(n))
    if g is not None:
        assert hashlib.sha256(b"".join(proof_res)).hexdigest() == g["sha256_proof"], "proof differs from the oracle digest"
        parity = "bit-exact: sha256(proof) equals the oracle's digest (tests/golden/sipp_large.json)"
    if world > 1:
        # the sharded proof must be byte-identical to the single-GPU proof of the same inputs (BASELINE config 3)
        assert b"".join(proof_res) == b"".join(sipp_b200.sipp_prove_native(A, B)), "sharded proof differs from the single-GPU proof"
    value = n * K / t_res
    e2e = n * K / t_e2e
    # Units of the Miller kernels: Miller loops their launches compute (pairs e(A_i, B_j) evaluated), each counted at the textbook
    # 9,008 Fq-mul (SURVEY 8d).  The pairing-matrix stages (SIPP_OPT_MATRIX_*) compute MORE loops than the reference's 3n - 2 --
    # block products of every pair of blocks, so that rounds become matrix folds -- and compute them cheaper (line coefficients of
    # a B point shared by all its partners, squarings shared by the pairs of a group); both ratios are reported.
    loops_step = st["miller_pairs"] / K
    mill_ach = st["miller_pairs"] * FQMUL_PER_MILLER * IMAD_PER_FQMUL / max(st["miller_ms"] * 1e-3, 1e-12)
    useful_ach = miller_loops_per_prove(n) * K * FQMUL_PER_MILLER * IMAD_PER_FQMUL / max(st["miller_ms"] * 1e-3, 1e-12)
    tr_head = (NCU_TRAFFIC.get("headline") or {}).get("kernels", {})
    dom = tr_head.get("k_accum") or {}
    roofline = {"bound": "imad", "kernel": "Miller-loop kernels of rank 0 in the timed proves: first stage k_qlines_batch + k_eval_lines_mat + k_accum "
                                           "(2^17 loops: the 32 x 32 block matrix of the inputs), later stages k_lines_wide + k_accum_eng",
                "achieved": mill_ach / 1e12,
                "peak": imad_peak / 1e12, "unit": "T IMAD/s", "frac": mill_ach / imad_peak,
                "units": "Miller loops computed by the launches x 9,008 Fq-mul x 264 IMAD (algorithmic count per loop)",
                "miller_loops_computed_per_step": loops_step, "miller_loops_of_the_reference_per_step": miller_loops_per_prove(n),
                "frac_reference_loops_only": useful_ach / imad_peak,
                "traffic": dom.get("largest_launch_dram_bytes"),
                "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of the largest k_accum launch (ncu --set full, profiles/ncu_traffic.json): "
                                "it reads the line table once (29,120 B per loop); algorithmic input is 192 B per pair",
                "algorithmic_input_bytes_per_pair": 192, "line_table_bytes_per_pair": 29120,
                "launches": int(st["miller_launches"]), "avg_launch_ms": st["miller_ms"] / max(1, st["miller_launches"]),
                "peak_source": "measured in this run (sipp_microbench: max of IMAD, 2 x IMAD.WIDE, lo/hi carry chain, all in "
                               "32x32 product halves/s); MEASURED_PEAKS.json has no integer peak",
                "kernel_time_share": {"miller_ms": st["miller_ms"] / K, "reduce_final_exp_ms": st["reduce_fe_ms"] / K, "fold_ms": st["fold_ms"] / K,
                                      "other_ms": st["other_ms"] / K, "host_transcript_exposed_ms": st["transcript_ms"] / K,
                                      "step_ms": t_res / K * 1e3,
                                      "note": "the first stage's kernels (~20 ms at n = 2^12) and the look-ahead folds run under the host's absorb chain "
                                              "or on a side stream: the classes overlap and do not add up to the step"},
                "fold_hbm_gbs": (st["fold_points"] * 576 / max(st["fold_ms"] * 1e-3, 1e-12)) / 1e9,
                "saturated": sat, "microbench": peaks}
    line = {"metric": "SIPP native prove throughput (pairings aggregated per second)", "value": value, "unit": "pairs/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": t_res / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32 limbs (254-bit modular integer)", "data": "synthetic",
            "config": {"workload": "SIPP native prover, n=2^%d pairs, %dxB200%s" % (log2(n), world, "" if world == 1 else " strided shards (2^%d pairs per GPU), "
                                   "NCCL all-gather of the partial products inside the library" % log2(n // world)),
                       "n": n, "seed": 2, "miller_loops_per_step": miller_loops_per_prove(n), "l2": "flushed between steps (256 MB write)",
                       "fe_normalisation": "exact", "fq12_transcript_order": "w-basis", "parity": parity,
                       "pairing_matrix_stages": {"tail": lib.sipp_get_option(_lib.OPT_MATRIX_TAIL), "block_n": lib.sipp_get_option(_lib.OPT_MATRIX_BLOCK_N),
                                                 "block_r": lib.sipp_get_option(_lib.OPT_MATRIX_BLOCK_R), "first": lib.sipp_get_option(_lib.OPT_MATRIX_FIRST)},
                       "nccl_version": lib.sipp_comm_nccl_version() if world > 1 else None,
                       "host_transcript": {"poseidon_backend": {2: "AVX-512 IFMA", 1: "AVX-512", 0: "portable"}.get(lib.sipp_poseidon_backend()),
                                           "ns_per_permutation": lib.sipp_poseidon_ns_per_permutation(200000),
                                           "permutations_per_prove": 8 * n + 13 + 27 * log2(n),
                                           "note": "strictly serial chain on rank 0's host (prover_native.rs:36-39, transcript_native.rs:25-30); "
                                                   "measured in this run on this box's CPU"}},
            "prove_s": t_res / K, "miller_loops_per_s_per_gpu": miller_loops_per_prove(n) * K / t_res / world,
            "e2e": {"value": e2e, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": t_e2e / K * 1e3,
                    "note": "h2d summed over the ranks; rank 0 additionally reads the full host copy of A, B for the transcript (no device traffic)"},
            "gpu_launches": int(st["launches"]), "clocks": clk, "roofline": roofline}

    if not args.no_cpu_baseline and world == 1:
        from oracle import pyoracle as o
        sample_n = 256
        As, Bs = A[:64 * sample_n], B[:128 * sample_n]
        t0 = time.perf_counter()
        ref = o.sipp_prove(As, Bs, o.FAITHFUL, 1)
        dt = time.perf_counter() - t0
        t0 = time.perf_counter()
        o.sipp_prove(As, Bs, 0, os.cpu_count() or 1)
        dt_fast = time.perf_counter() - t0
        gpu = b"".join(sipp_b200.sipp_prove_native(As, Bs))
        assert gpu == ref, "GPU proof differs from the oracle on the baseline sample"
        line["cpu_baseline"] = {"value": sample_n / dt, "unit": "pairs/s", "cores": 1, "kind": "port",
                                "sample": "single-thread faithful restatement (one full pairing per pair) proving the first %d of the %d pairs, "
                                          "%.1f s; GPU proof of the same sample is byte-identical" % (sample_n, n, dt),
                                "all_cores_fast_variant": {"value": sample_n / dt_fast, "cores": os.cpu_count() or 1,
                                                           "note": "product of Miller loops + one final exponentiation, pthreads"}}
    if world == 1 and not args.quick:
        # the verifier of the same statement (verifier_native.rs:14-85: transcript replay, folds, GT updates, final pairing) through
        # the public call with host buffers
        sipp_b200.sipp_verify_native(A, B, proof_res)
        tv = []
        for _ in range(3):
            t0 = time.perf_counter()
            sipp_b200.sipp_verify_native(A, B, proof_res)
            tv.append(time.perf_counter() - t0)
        line["verify"] = {"ms": min(tv) * 1e3, "unit": "ms per sipp_verify_native of the timed proof (host buffers, best of 3)",
                          "pairs_per_s": n / min(tv)}
    if args.quick:
        line["e2e"] = None
        line["config"]["quick"] = "one warm-up step, e2e leg skipped (--quick)"
    if large:
        line["baseline_configs"] = large
    if bm is not None:
        bst = bm["stats"]
        line["batched_instances"] = {"workload": "%d independent n=128 instances over %d GPU(s), lock-step, transcripts on the device, instances sharded by "
                                                 "rank (no collective)" % (args.batch_instances, world),
                                     "instances_per_s": args.batch_instances / bm["t_res"], "e2e_instances_per_s": args.batch_instances / bm["t_e2e"],
                                     "pairs_per_s": args.batch_instances * 128 / bm["t_res"], "ms": bm["t_res"] * 1e3,
                                     "rank0_miller_ms": bst["miller_ms"], "rank0_final_exp_ms": bst["reduce_fe_ms"], "rank0_fold_ms": bst["fold_ms"],
                                     "miller_frac_of_imad_peak": bst["miller_pairs"] * FQMUL_PER_MILLER * IMAD_PER_FQMUL
                                     / max(bst["miller_ms"] * 1e-3, 1e-12) / imad_peak}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"proof": b"".join(proof_res), **large_proofs}, bm["proofs"] if bm is not None else None)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
