"""Both alternatives of the two open conventions, and the option values and shapes that change which kernels run, end to end on
the GPU against the CPU oracle.

H1 (SIPP_OPT_FE_NORMALISATION: exact exponent or arkworks' multiple) and H2 (SIPP_OPT_FQ12_ORDER: w-basis or nested order of the
transcript's Fq12) cannot be settled offline (DESIGN.md §2).  Each convention is one bit of the oracle's `opts` (oracle.FE_ARK,
oracle.FQ12_NESTED), pinned to the pure-Python model in tests/test_oracle_conventions.py; every test below compares the GPU with
the oracle under the same bits: single proofs on every stage route, the round-granular API with a host transcript, the verifier
(single and batched), the batched prover and the sharded prover.

The second half runs, under the default convention, the option values and shapes no other test reaches: explicit first-stage
budgets (SIPP_OPT_MATRIX_FIRST = 10..24), the throughput ("big") matrix build inside look-ahead stages, sub-batches on their own
streams, the chunked line table of a large batch, and the entry points the benchmark times.  Each of them asserts that its
branch was taken (stage blocks from the host-side policy, Miller launch counts), so that a later change of a threshold cannot
turn it into a no-op."""
import ctypes
import math
import os
import socket
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
THREADS = os.cpu_count() or 1

# every option of include/sipp_b200.h with its default
DEFAULTS = {1: 0, 2: 0, 3: 0, 4: 1, 5: 8192, 6: 1, 7: 256, 8: 1536, 9: 32, 10: 1, 11: 0, 12: 1, 13: 1, 14: 32, 15: 256, 16: 8, 17: 1}
OPT_FE_NORMALISATION, OPT_FQ12_ORDER, OPT_PROFILE, OPT_PIPELINE, OPT_WIDE_LINES_MAX, OPT_FE_ENGINE, OPT_WIDE_FOLD_MAX, OPT_WIDE_ACCUM_MAX = 1, 2, 3, 4, 5, 6, 7, 8
OPT_BATCH_STREAMS, OPT_BATCH_QLINES, OPT_MATRIX_TAIL, OPT_MATRIX_BLOCK_N, OPT_MATRIX_BLOCK_R, OPT_MATRIX_FIRST = 11, 12, 14, 15, 16, 17
CONVENTIONS = (0, 1, 2, 3)   # bit 0: arkworks normalisation (oracle.FE_ARK), bit 1: nested Fq12 order (oracle.FQ12_NESTED)

# the line table of one pair (91 lines x 80 words x 4 B) and the line-table budget of one batched call (batch.cu)
LINES_BYTES_PER_PAIR = 91 * 80 * 4
BATCH_LINES_CAP = 1 << 34


@pytest.fixture(scope="module")
def sipp():
    import sipp_b200
    from sipp_b200 import _lib
    _lib.require_gpu_once()
    return sipp_b200


@pytest.fixture(scope="module")
def lib(sipp):
    from sipp_b200 import _lib
    return _lib.load()


@pytest.fixture(autouse=True)
def options(lib):
    """every test starts from the defaults, whatever earlier tests left, and leaves the options as it found them"""
    from sipp_b200 import _lib
    saved = {o: lib.sipp_get_option(o) for o in DEFAULTS}
    try:
        for o, v in DEFAULTS.items():
            _lib.check(lib.sipp_set_option(o, v))
        yield
    finally:
        for o, v in saved.items():
            _lib.check(lib.sipp_set_option(o, v))


def set_convention(sipp, opts):
    sipp.set_option(OPT_FE_NORMALISATION, opts & 1)
    sipp.set_option(OPT_FQ12_ORDER, opts >> 1)


@pytest.fixture(params=[1, 2, 3], ids=["ark-normalisation", "nested-order", "ark-nested"])
def convention(request, sipp, options):
    set_convention(sipp, request.param)
    return request.param


def inst(X, size, n, j):
    """instance j of a batch: pairs [j n, (j + 1) n)"""
    return X[size * n * j:size * n * (j + 1)]


def joined(proofs):
    return [b"".join(p) for p in proofs]


def stage_plan(lib, n):
    """the stages a single proof of n points runs through, from the host-side policy (sipp_test_stage_blocks): ("first", nr) for
    a first stage of nr blocks over the inputs, ("ahead", nr) for a look-ahead stage, ("tail", points) for the matrix of single
    points, ("points", count) for rounds on the points"""
    plan, nr = [], lib.sipp_test_stage_blocks(0, n)
    if nr:
        plan.append(("first", nr) if nr < n else ("tail", n))
        n //= nr
    while n > 1:
        nr = lib.sipp_test_stage_blocks(1, n)
        if nr == n:
            plan.append(("tail", n))
            break
        if nr:
            plan.append(("ahead", nr))
            n //= nr
        else:
            if plan and plan[-1][0] == "points":
                plan[-1] = ("points", plan[-1][1] + 1)
            else:
                plan.append(("points", 1))
            n //= 2
    return plan


def matrix_build(n, nr):
    """what mat_build_ex (sipp_b200.cu) runs for a stage of nr blocks over n points: ("small", 1) = the lane engines, ("big", kpg) =
    k_qlines_batch + k_eval_lines_mat + k_accum with kpg pairs of a block per accumulator group"""
    m, pairs = n // nr, n * nr
    if not (m > 1 and pairs > 8192):
        return "small", 1
    return "big", max(1, min((m + 19) // 20, (pairs + 11839) // 11840))


# ---- A. single proofs under each convention ------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,plan", [
    (1, []),                                                   # a proof of Z only
    (2, [("tail", 2)]),                                        # the whole proof on the matrix of its inputs
    (16, [("tail", 16)]),
    (64, [("first", 8), ("tail", 8)]),
    (256, [("first", 8), ("tail", 32)]),
    (1024, [("first", 8), ("ahead", 8), ("tail", 16)]),        # small first-stage build, a look-ahead stage
    (2048, [("first", 16), ("ahead", 8), ("tail", 16)]),       # big first-stage build (kpg 3, ragged last group)
])
def test_prove_under_convention(sipp, lib, oracle, convention, n, plan):
    assert stage_plan(lib, n) == plan
    if n == 1024:
        assert matrix_build(n, 8) == ("small", 1)
    if n == 2048:
        assert matrix_build(n, 16) == ("big", 3) and (n // 16) % 3
    A, B = sipp.seeded_inputs(700 + n, n)
    proof = b"".join(sipp.sipp_prove_native(A, B))
    assert proof == oracle.sipp_prove(A, B, convention, threads=THREADS)
    if convention & 1 or n >= 4:                               # the order shows from the second challenge on: up to n = 2
        assert proof != oracle.sipp_prove(A, B, 0, threads=THREADS)   # no challenge enters the proof


def _exceptional_n64(oracle):
    """identity in G1, identity in G2, equal points in the two halves (as in test_matrix_tail_thresholds)"""
    A, B = oracle.seeded_inputs(77, 64, threads=THREADS)
    A = bytearray(A); B = bytearray(B)
    A[64 * 5:64 * 6] = bytes(64)
    B[128 * 41:128 * 42] = bytes(128)
    A[64 * 9:64 * 10] = A[64 * 41:64 * 42]
    return bytes(A), bytes(B)


def test_prove_exceptional_inputs_under_convention(sipp, oracle, convention):
    A, B = _exceptional_n64(oracle)
    assert b"".join(sipp.sipp_prove_native(A, B)) == oracle.sipp_prove(A, B, convention, threads=THREADS)


@pytest.mark.parametrize("pipeline", [(1, 8192, 1), (1, 0, 0), (0, 0, 0)], ids=["split-engines", "split-thread-lines-coop-fe", "per-thread"])
def test_prove_pipelines_ark_nested(sipp, lib, oracle, pipeline):
    """n = 64 under both alternatives on every Miller pipeline (the settings of test_gpu_parity.py's `pipeline` fixture); with the
    engines off the matrix stages are off too, so the last two are the point-fold routes"""
    set_convention(sipp, 3)
    sipp.set_option(OPT_PIPELINE, pipeline[0])
    sipp.set_option(OPT_WIDE_LINES_MAX, pipeline[1])
    sipp.set_option(OPT_FE_ENGINE, pipeline[2])
    sipp.set_option(OPT_WIDE_FOLD_MAX, 1 << 20 if pipeline[2] else 0)
    sipp.set_option(OPT_WIDE_ACCUM_MAX, 8192 if pipeline[2] else 0)
    assert stage_plan(lib, 64) == ([("first", 8), ("tail", 8)] if pipeline[2] else [("points", 6)])
    A, B = _exceptional_n64(oracle)
    assert b"".join(sipp.sipp_prove_native(A, B)) == oracle.sipp_prove(A, B, 3, threads=THREADS)


def test_round_api_host_transcript_under_convention(sipp, lib, oracle, convention):
    """a host that keeps its own sipp.Transcript and drives the stages round by round: every challenge is the oracle's"""
    n = 128
    assert stage_plan(lib, n) == [("first", 8), ("tail", 16)]
    A, B = oracle.seeded_inputs(1, n, threads=THREADS)
    want, trace = oracle.sipp_prove(A, B, convention, threads=THREADS, trace=True)
    ctx = sipp.ProverContext(A, B)
    try:
        ctx.set_stages(True)
        tr = sipp.Transcript()
        proof = [ctx.inner_product()]
        for i in range(n):
            tr.append_g1(A[64 * i:64 * i + 64]); tr.append_g2(B[128 * i:128 * i + 128])
        tr.append_fq12(proof[0])
        rnd = 0
        while len(ctx) > 1:
            zl, zr = ctx.cross_products()
            proof += [zl, zr]
            tr.append_fq12(zl); tr.append_fq12(zr)
            x = tr.get_challenge()
            assert x == trace["challenges"][32 * rnd:32 * rnd + 32], rnd
            ctx.fold(x, sipp.fr_inverse(x))
            rnd += 1
        assert rnd == 7
        proof.reverse()
        assert b"".join(proof) == want
    finally:
        ctx.close()


@pytest.mark.parametrize("fe_engine", [1, 0], ids=["batched-gt-updates", "gt-fold-per-round"])
@pytest.mark.parametrize("n", [16, 256])
def test_verify_under_convention(sipp, oracle, convention, n, fe_engine):
    sipp.set_option(OPT_FE_ENGINE, fe_engine)
    A, B = oracle.seeded_inputs(800 + n, n, threads=THREADS)
    proof = oracle.sipp_prove(A, B, convention, threads=THREADS)
    st = sipp.sipp_verify_native(A, B, [proof[i:i + 384] for i in range(0, len(proof), 384)])
    ok, want = oracle.sipp_verify(A, B, proof, convention, threads=THREADS)
    assert ok
    assert (st.final_A, st.final_B, st.final_Z) == (want["final_A"], want["final_B"], want["final_Z"])
    assert st.Z == proof[-384:]


def test_verify_accepts_only_its_own_convention(sipp, oracle):
    """a proof made under convention a verifies under b if and only if a == b (GPU prover and verifier, n = 16)"""
    n = 16
    A, B = oracle.seeded_inputs(816, n, threads=THREADS)
    proofs = {}
    for a in CONVENTIONS:
        set_convention(sipp, a)
        proofs[a] = sipp.sipp_prove_native(A, B)
        assert b"".join(proofs[a]) == oracle.sipp_prove(A, B, a, threads=THREADS)
    for a in CONVENTIONS:
        for b in CONVENTIONS:
            set_convention(sipp, b)
            if a == b:
                sipp.sipp_verify_native(A, B, proofs[a])
            else:
                with pytest.raises(sipp.VerificationError):
                    sipp.sipp_verify_native(A, B, proofs[a])


# ---- B. batched prover and verifier under each convention ----------------------------------------------------------------------
@pytest.mark.parametrize("n,count", [(1, 5), (16, 33), (128, 64), (8, 1024)])
def test_batch_under_convention(sipp, oracle, convention, n, count):
    """every instance == the single-instance GPU proof; the first two and the last == the oracle; the batched verifier's statements
    == the oracle's.  (8, 1024): the 2,048 cross products of a round are more than 12 per SM, so they take the 6-lane final
    exponentiation (launch_fe_batch) instead of the 32-lane machines"""
    if (n, count) == (8, 1024):
        import torch
        assert 2 * count > 12 * torch.cuda.get_device_properties(0).multi_processor_count
    A, B = sipp.seeded_inputs(900 + n, n * count)
    proofs = sipp.sipp_prove_native_batch(A, B, n)
    assert len(proofs) == count
    for j in range(count):
        assert proofs[j] == sipp.sipp_prove_native(inst(A, 64, n, j), inst(B, 128, n, j)), j
    sts = sipp.sipp_verify_native_batch(A, B, n, proofs)
    assert not any(isinstance(s, Exception) for s in sts)
    for j in (0, 1, count - 1):
        a, b = inst(A, 64, n, j), inst(B, 128, n, j)
        assert b"".join(proofs[j]) == oracle.sipp_prove(a, b, convention, threads=THREADS), j
        ok, want = oracle.sipp_verify(a, b, b"".join(proofs[j]), convention, threads=THREADS)
        assert ok and (sts[j].final_A, sts[j].final_B, sts[j].final_Z) == (want["final_A"], want["final_B"], want["final_Z"]), j


def test_batch_verify_accepts_only_its_own_convention(sipp, oracle):
    """per instance: a batch of proofs made under convention a verifies under b if and only if a == b"""
    n, count = 16, 33
    A, B = sipp.seeded_inputs(933, n * count)
    proofs = {}
    for a in CONVENTIONS:
        set_convention(sipp, a)
        proofs[a] = sipp.sipp_prove_native_batch(A, B, n)
        assert b"".join(proofs[a][count - 1]) == oracle.sipp_prove(inst(A, 64, n, count - 1), inst(B, 128, n, count - 1), a, threads=THREADS)
    for a in CONVENTIONS:
        for b in CONVENTIONS:
            set_convention(sipp, b)
            sts = sipp.sipp_verify_native_batch(A, B, n, proofs[a])
            assert [isinstance(s, sipp.VerificationError) for s in sts] == [a != b] * count, (a, b)


# ---- C. sharded prover under both alternatives ---------------------------------------------------------------------------------
def _sharded_worker(rank, world, port, n, seed, opts, q):
    sys.path.insert(0, ROOT)
    try:
        import torch
        import torch.distributed as dist
        import sipp_b200
        from sipp_b200 import _lib, sharded
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        os.environ["SIPP_DEVICE"] = "0"
        dist.init_process_group("gloo", rank=rank, world_size=world)
        lib = _lib.load()
        _lib.require_gpu(0)
        sipp_b200.set_option(OPT_FE_NORMALISATION, opts & 1)   # every rank: the ranks' partial products and rank 0's exponentiations
        sipp_b200.set_option(OPT_FQ12_ORDER, opts >> 1)

        def allgather(_u, send, recv, nbytes):
            t = torch.frombuffer(bytearray(ctypes.string_at(send, nbytes)), dtype=torch.uint8)
            out = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(out, t)
            ctypes.memmove(recv, b"".join(x.numpy().tobytes() for x in out), nbytes * world)
            return 0

        def broadcast(_u, buf, nbytes, root):
            t = torch.frombuffer(bytearray(ctypes.string_at(buf, nbytes)), dtype=torch.uint8)
            dist.broadcast(t, src=root)
            ctypes.memmove(buf, t.numpy().tobytes(), nbytes)
            return 0
        keep = [_lib.ALLGATHER_FN(allgather), _lib.BROADCAST_FN(broadcast)]
        _lib.check(lib.sipp_comm_init_host(rank, world, keep[0], keep[1], None))
        A, B = sipp_b200.seeded_inputs(seed, n)
        Al, Bl = sharded.shard_points(A, B, rank, world)
        proof = sharded.sharded_prove(Al, Bl, n, A if rank == 0 else None, B if rank == 0 else None)
        q.put((rank, None if proof is None else b"".join(proof), A, B))
        dist.barrier()
        lib.sipp_comm_destroy()
        dist.destroy_process_group()
    except Exception as e:  # noqa: BLE001
        q.put((rank, "error: %r" % (e,), None, None))
        raise


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("n", [64, 2048])
def test_sharded_ark_nested(oracle, n):
    """world 2 on one GPU over host collectives, both options set in every rank"""
    import torch.multiprocessing as mp
    world, opts = 2, 3
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_sharded_worker, args=(r, world, port, n, 41, opts, q)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        got = {}
        for _ in range(world):
            item = q.get(timeout=600)
            got[item[0]] = item
        for p in procs:
            p.join(timeout=120)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join()
    _, proof, A, B = got[0]
    assert not isinstance(proof, str), proof
    assert got[1][1] is None
    assert proof == oracle.sipp_prove(A, B, opts, threads=THREADS)


# ---- D. option values and shapes that change kernels (default convention) -----------------------------------------------------
@pytest.fixture(scope="module")
def reference(sipp, oracle):
    """seeded inputs of n points and the oracle's proof under the default convention, computed once per n"""
    cache = {}

    def get(n):
        if n not in cache:
            A, B = sipp.seeded_inputs(1100 + n, n)
            cache[n] = (A, B, oracle.sipp_prove(A, B, 0, threads=THREADS))
        return cache[n]
    return get


@pytest.mark.parametrize("n,first,nr,build", [
    (512, 11, 4, ("small", 1)), (512, 12, 8, ("small", 1)), (512, 13, 16, ("small", 1)),
    (1024, 14, 16, ("big", 2)), (1024, 15, 32, ("big", 2)),
    (2048, 13, 4, ("small", 1)), (2048, 14, 8, ("big", 2)), (2048, 15, 16, ("big", 3)), (2048, 16, 32, ("big", 4)),
])
def test_first_stage_budget(sipp, lib, reference, n, first, nr, build):
    """SIPP_OPT_MATRIX_FIRST = 10..24: a first stage of 2^first Miller loops whatever n (kept at or below 2^16: 1.9 GB of lines)"""
    sipp.set_option(OPT_MATRIX_FIRST, first)
    assert lib.sipp_get_option(OPT_MATRIX_FIRST) == first
    assert lib.sipp_test_stage_blocks(0, n) == nr and nr * n <= 1 << first
    assert matrix_build(n, nr) == build
    if build == ("big", 3):
        assert (n // nr) % 3                                   # the last accumulator group of a block is ragged
    A, B, want = reference(n)
    assert b"".join(sipp.sipp_prove_native(A, B)) == want


@pytest.mark.parametrize("lead", [0, 1], ids=["from-inputs", "after-a-point-fold"])
@pytest.mark.parametrize("n,r,kpg", [(1024, 16, 2), (1024, 32, 2), (2048, 8, 2), (2048, 16, 3), (2048, 32, 4), (512, 32, 1)])
def test_big_lookahead_stage(sipp, lib, reference, n, r, kpg, lead):
    """a look-ahead stage large enough for the throughput build (more than 8,192 Miller loops): SIPP_OPT_MATRIX_FIRST = 0,
    SIPP_OPT_MATRIX_BLOCK_N >= n.  With `lead` the proof has 2n points and its first round runs on the points, so the stage is
    built from folded points while the next folds run on the side stream"""
    total = n << lead
    sipp.set_option(OPT_MATRIX_FIRST, 0)
    sipp.set_option(OPT_MATRIX_BLOCK_N, 4096 if not lead else n)
    sipp.set_option(OPT_MATRIX_BLOCK_R, r)
    plan = stage_plan(lib, total)
    assert plan[:1 + lead] == ([("points", 1)] if lead else []) + [("ahead", r)], plan
    assert matrix_build(n, r) == ("big", kpg)
    if kpg == 3:
        assert (n // r) % 3
    A, B, want = reference(total)
    assert b"".join(sipp.sipp_prove_native(A, B)) == want


@pytest.fixture(scope="module")
def streams_reference(sipp, oracle):
    """a batch of `count` instances of n = 32 proved as one batch (SIPP_OPT_BATCH_STREAMS = 0), sampled against the oracle"""
    cache = {}

    def get(count):
        if count not in cache:
            n = 32
            A, B = sipp.seeded_inputs(1200 + count, n * count)
            sipp.stats(reset=True)
            proofs = joined(sipp.sipp_prove_native_batch(A, B, n))
            assert sipp.stats()["miller_launches"] == 6             # one sub-batch: Z + 5 rounds
            for j in (0, count * 3 // 8, count - 1):
                assert proofs[j] == oracle.sipp_prove(inst(A, 64, n, j), inst(B, 128, n, j), threads=THREADS), j
            cache[count] = (A, B, proofs)
        return cache[count]
    return get


@pytest.mark.parametrize("count,streams,profile,nsub", [(64, 2, 0, 2), (128, 4, 0, 4), (300, 8, 0, 8), (100, 8, 0, 2), (300, 8, 1, 1)])
def test_batch_streams(sipp, streams_reference, count, streams, profile, nsub):
    """SIPP_OPT_BATCH_STREAMS: sub-batches of at least 32 instances on their own streams (300 / 8: slices of 37 or 38);
    SIPP_OPT_PROFILE = 1 forces one sub-batch"""
    n = 32
    A, B, want = streams_reference(count)
    sipp.set_option(OPT_BATCH_STREAMS, streams)
    sipp.set_option(OPT_PROFILE, profile)
    sipp.stats(reset=True)
    got = joined(sipp.sipp_prove_native_batch(A, B, n))
    assert sipp.stats()["miller_launches"] == nsub * (int(math.log2(n)) + 1)
    assert got == want


def _chunks(nproducts, h):
    """products per launch of one round of a batch whose line table is the whole budget"""
    pc = BATCH_LINES_CAP // (h * LINES_BYTES_PER_PAIR)
    return [min(pc, nproducts - p0) for p0 in range(0, nproducts, pc)]


@pytest.fixture(scope="module")
def chunked_reference(sipp, oracle):
    """n = 128, 4,736 instances (606,208 pairs), and the proofs of its two halves of 2,368 instances, each one unchunked batch
    (computed on first use)"""
    cache = []

    def get():
        if not cache:
            n, count = 128, 4736
            A, B = sipp.seeded_inputs(13, n * count)
            h = count // 2
            proofs = []
            for k in range(2):
                sipp.stats(reset=True)
                proofs += joined(sipp.sipp_prove_native_batch(inst(A, 64, n * h, k), inst(B, 128, n * h, k), n))
                assert sipp.stats()["miller_launches"] == int(math.log2(n)) + 1
            for j in (0, 4608, 4609, 4610, 4735):
                assert proofs[j] == oracle.sipp_prove(inst(A, 64, n, j), inst(B, 128, n, j), threads=THREADS), j
            cache.append((A, B, proofs))
        return cache[0]
    return get


@pytest.mark.parametrize("qlines", [1, 0], ids=["shared-qlines", "lines-per-pair"])
def test_batch_chunked_line_table(sipp, chunked_reference, qlines):
    """a batch whose line table exceeds the 16 GiB budget runs each of its first rounds in several launches (products p0.. of
    the round, partials at p0 x groups per product): Z in 4,609 + 127 products, round 1 in 9,218 + 254"""
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < 40 << 30:
        pytest.skip("needs about 28 GB of device memory (40 GB free asked for on a shared GPU); %.1f GB free" % (free / 2**30))
    n, count = 128, 4736
    assert _chunks(count, n) == [4609, 127]
    assert _chunks(2 * count, n // 2) == [9218, 254]
    rounds = int(math.log2(n))
    launches = len(_chunks(count, n)) + sum(len(_chunks(2 * count, n >> k)) for k in range(1, rounds + 1))
    assert launches == rounds + 1 + 2                          # unchunked: Z + one launch per round
    if qlines:
        assert n * count * 91 * 48 * 4 <= BATCH_LINES_CAP      # the Q-only lines of every B point fit the budget: they are shared
    A, B, want = chunked_reference()
    sipp.set_option(OPT_BATCH_QLINES, qlines)
    sipp.stats(reset=True)
    got = joined(sipp.sipp_prove_native_batch(A, B, n))
    assert sipp.stats()["miller_launches"] == launches
    assert len(got) == count
    bad = [j for j in range(count) if got[j] != want[j]]
    assert not bad, "%d instances differ, first %s" % (len(bad), bad[:8])


def test_batch_device_entry(sipp, lib):
    """sipp_prove_native_batch_device (the resident timing of bench.py) on torch buffers == sipp_prove_native_batch, 512 x n = 128"""
    import torch
    from sipp_b200 import _lib
    n, count = 128, 512
    A, B = sipp.seeded_inputs(5, n * count)
    plen = lib.sipp_proof_len(n)
    dA = torch.frombuffer(bytearray(A), dtype=torch.uint8).cuda()
    dB = torch.frombuffer(bytearray(B), dtype=torch.uint8).cuda()
    dP = torch.zeros(count * plen * 384, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    _lib.check(lib.sipp_prove_native_batch_device(dA.data_ptr(), dB.data_ptr(), n, count, dP.data_ptr()))
    torch.cuda.synchronize()
    got = dP.cpu().numpy().tobytes()
    assert got == b"".join(joined(sipp.sipp_prove_native_batch(A, B, n)))


def test_sharded_device_entry_world_one_profiled(sipp, lib):
    """sharded_prove from device buffers without a communicator (bench.py's headline path: a world of one), under
    SIPP_OPT_PROFILE = 1 as in the timed steps, == the committed oracle proof of n = 2^12, seed 2"""
    import torch
    from sipp_b200 import sharded
    n = 1 << 12
    assert lib.sipp_comm_world() == 1
    A, B = sipp.seeded_inputs(2, n)
    dA = torch.frombuffer(bytearray(A), dtype=torch.uint8).cuda()
    dB = torch.frombuffer(bytearray(B), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    sipp.set_option(OPT_PROFILE, 1)
    sipp.stats(reset=True)
    proof = sharded.sharded_prove(None, None, n, A, B, device_ptrs=(dA.data_ptr(), dB.data_ptr()))
    assert sipp.stats()["miller_ms"] > 0                       # the profile spans were recorded
    with open(os.path.join(HERE, "golden", "sipp_large_seed2_n2p12.proof.bin"), "rb") as f:
        assert b"".join(proof) == f.read()
