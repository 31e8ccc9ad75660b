"""The library's sharded prover (`sipp_prove_native_sharded`, sipp_b200/csrc/sharded.cu) through the C ABI, on real GPUs.

* several ranks on ONE GPU, collectives over the host-memory callbacks (`sipp_comm_init_host`, gloo underneath): the CUDA
  backend's partial products, in-place gather slots, challenge broadcast, local folds and the tail collapse run exactly as
  they do over NCCL, so the single-GPU box checks them bit for bit against the oracle;
* one rank per GPU over NCCL (`sipp_comm_init`) when the box has at least two GPUs."""
import ctypes
import os
import sys

import pytest
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, n, seed, mode, q):
    sys.path.insert(0, ROOT)
    try:
        import torch
        import torch.distributed as dist
        from sipp_b200 import _lib, sharded
        import sipp_b200
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        dev = rank if mode == "nccl" else 0
        os.environ["SIPP_DEVICE"] = str(dev)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        lib = _lib.load()
        _lib.require_gpu(dev)
        keep = []
        if mode == "nccl":
            sharded.comm_init_torch()
        else:
            def allgather(_u, send, recv, nbytes):
                t = torch.frombuffer(bytearray(ctypes.string_at(send, nbytes)), dtype=torch.uint8)
                out = [torch.empty_like(t) for _ in range(world)]
                dist.all_gather(out, t)
                ctypes.memmove(recv, b"".join(bytes(x.numpy().tobytes()) for x in out), nbytes * world)
                return 0

            def broadcast(_u, buf, nbytes, root):
                t = torch.frombuffer(bytearray(ctypes.string_at(buf, nbytes)), dtype=torch.uint8)
                dist.broadcast(t, src=root)
                ctypes.memmove(buf, bytes(t.numpy().tobytes()), nbytes)
                return 0
            keep = [_lib.ALLGATHER_FN(allgather), _lib.BROADCAST_FN(broadcast)]
            _lib.check(lib.sipp_comm_init_host(rank, world, keep[0], keep[1], None))
        assert lib.sipp_comm_rank() == rank and lib.sipp_comm_world() == world
        A, B = sipp_b200.seeded_inputs(seed, n)
        Al, Bl = sharded.shard_points(A, B, rank, world)
        proof = sharded.sharded_prove(Al, Bl, n, A if rank == 0 else None, B if rank == 0 else None)
        # the same from a shard resident in HBM
        dA = torch.frombuffer(bytearray(Al), dtype=torch.uint8).cuda(dev)
        dB = torch.frombuffer(bytearray(Bl), dtype=torch.uint8).cuda(dev)
        proof2 = sharded.sharded_prove(None, None, n, A if rank == 0 else None, B if rank == 0 else None, device_ptrs=(dA.data_ptr(), dB.data_ptr()))
        # a rank whose shard does not decode must end every rank with an error, not leave the others in a collective
        bad = bytearray(Al)
        if rank == world - 1:
            bad[0:32] = b"\xff" * 32
        rc = lib.sipp_prove_native_sharded(bytes(bad), Bl, n, A if rank == 0 else None, B if rank == 0 else None,
                                           ctypes.create_string_buffer(384 * lib.sipp_proof_len(n)) if rank == 0 else None)
        q.put((rank, None if proof is None else b"".join(proof), None if proof2 is None else b"".join(proof2), rc, A, B))
        dist.barrier()
        lib.sipp_comm_destroy()
        dist.destroy_process_group()
    except Exception as e:  # noqa: BLE001
        q.put((rank, "error: %r" % (e,), None, 0, None, None))
        raise


def _run(world, n, seed, mode, oracle):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + (os.getpid() % 1000) + world * 11 + (n % 97)
    procs = [ctx.Process(target=_worker, args=(r, world, port, n, seed, mode, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = {}
    for _ in range(world):
        item = q.get(timeout=600)
        got[item[0]] = item
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    _, proof, proof2, rc0, A, B = got[0]
    assert not isinstance(proof, str), proof
    want = oracle.sipp_prove(A, B, 0, os.cpu_count() or 1)
    assert proof == want, "sharded proof differs from the oracle"
    assert proof2 == want, "sharded proof from device-resident shards differs from the oracle"
    for r in range(world):
        assert got[r][3] == -6, "rank %d: a shard that does not decode must fail every rank with SIPP_ERR_ENCODING (got %d)" % (r, got[r][3])
        if r:
            assert got[r][1] is None


@pytest.mark.parametrize("world,n", [(2, 64), (4, 64), (2, 2), (4, 4), (2, 2048), (8, 8)])
def test_sharded_on_one_gpu_host_collectives(world, n, oracle):
    _run(world, n, 31, "host", oracle)


@pytest.mark.parametrize("n", [2, 256, 4096])
def test_sharded_nccl(n, oracle):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (one rank per GPU over NCCL)")
    world = 1
    while world * 2 <= min(torch.cuda.device_count(), 8):
        world *= 2
    for w in sorted({2, world}):
        if n >= w:
            _run(w, n, 32, "nccl", oracle)


def test_sharded_without_communicator_is_single_gpu(oracle):
    import sipp_b200
    from sipp_b200 import _lib, sharded
    _lib.require_gpu_once()
    A, B = oracle.seeded_inputs(33, 32)
    assert b"".join(sharded.sharded_prove(A, B, 32, A, B)) == oracle.sipp_prove(A, B) == b"".join(sipp_b200.sipp_prove_native(A, B))
