"""Multi-GPU SIPP prover: a ctypes wrapper of the library's sharded prover (sipp_b200/csrc/sharded.cu).

One process per GPU; rank g owns the pairs i = g (mod world).  The protocol loop (prover_native.rs:26-80 over the ranks),
the NCCL all-gather of the 384-byte partial products and the challenge broadcast all live inside libsipp_b200.so --
this module only slices inputs, ships the NCCL unique id with whatever the host already has (torch.distributed here)
and calls `sipp_prove_native_sharded`.  There is no CPU fallback.
"""
import ctypes
from typing import List, Optional

from . import _lib

G1_BYTES, G2_BYTES, FQ12_BYTES = 64, 128, 384


def shard_indices(n: int, rank: int, world: int) -> List[int]:
    """global indices owned by `rank`: i = rank (mod world)"""
    return list(range(rank, n, world))


def shard_points(A: bytes, B: bytes, rank: int, world: int):
    n = len(A) // G1_BYTES
    idx = shard_indices(n, rank, world)
    return (b"".join(A[G1_BYTES * i:G1_BYTES * (i + 1)] for i in idx),
            b"".join(B[G2_BYTES * i:G2_BYTES * (i + 1)] for i in idx))


def shard_instances(count: int, rank: int, world: int):
    """Batched instances (BASELINE config 5) are independent: rank g proves the contiguous slice [lo, hi) of the instances
    and no collective is needed.  Slices differ by at most one instance."""
    base, extra = divmod(count, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def shard_instances_ragged(lengths, rank: int, world: int):
    """Ragged batches (sipp_prove_native_batch_ragged): rank g proves the contiguous slice [lo, hi) of the instances.  The slices
    are balanced by the pairs of the products, sum_j (3 n_j - 2), not by instance count: slice g ends at the instance boundary
    whose running cost is nearest to (g + 1) / world of the total (the first such boundary on a tie)."""
    prefix = [0]
    for n in lengths:
        prefix.append(prefix[-1] + 3 * int(n) - 2)

    def cut(g):
        target = prefix[-1] * g
        return min(range(len(prefix)), key=lambda j: (abs(prefix[j] * world - target), j))
    return cut(rank), cut(rank + 1)


def comm_init_nccl(rank: int, world: int, broadcast_bytes) -> None:
    """NCCL communicator inside the library.  `broadcast_bytes(b: Optional[bytes]) -> bytes` ships rank 0's 128-byte unique id
    to every rank over the host's own channel (e.g. `comm_init_torch` below)."""
    _lib.require_gpu_once()
    lib = _lib.load()
    uid = ctypes.create_string_buffer(128)
    if rank == 0:
        _lib.check(lib.sipp_comm_get_unique_id(uid))
    uid = broadcast_bytes(uid.raw if rank == 0 else None)
    _lib.check(lib.sipp_comm_init(uid, rank, world))


def comm_init_torch() -> None:
    """unique id shipped over the already-initialised torch.distributed group"""
    import torch.distributed as dist

    def bcast(b):
        box = [b]
        dist.broadcast_object_list(box, src=0)
        return box[0]
    comm_init_nccl(dist.get_rank(), dist.get_world_size(), bcast)


def sharded_prove(A_local, B_local, n: int, A_full: Optional[bytes] = None, B_full: Optional[bytes] = None,
                  device_ptrs=None) -> Optional[List[bytes]]:
    """Collective call: every rank passes its strided shard (host bytes, or `device_ptrs` = (dA, dB) already in HBM) and the
    total n; rank 0 also passes the full A, B (the transcript absorbs every point) and gets the proof, the others None."""
    lib = _lib.load()
    rank0 = lib.sipp_comm_rank() == 0
    proof = ctypes.create_string_buffer(FQ12_BYTES * lib.sipp_proof_len(n)) if rank0 else None
    if device_ptrs is None:
        a, b = (x if isinstance(x, ctypes.c_char_p) else bytes(x) for x in (A_local, B_local))   # c_char_p: e.g. pinned host memory
        _lib.check(lib.sipp_prove_native_sharded(a, b, n, A_full, B_full, proof))
    else:
        _lib.check(lib.sipp_prove_native_sharded_device(device_ptrs[0], device_ptrs[1], n, A_full, B_full, proof))
    return [proof.raw[i:i + FQ12_BYTES] for i in range(0, len(proof.raw), FQ12_BYTES)] if rank0 else None
