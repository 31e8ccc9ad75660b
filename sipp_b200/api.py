"""Host-side mirror of the reference's native SIPP interface, on top of the C ABI.

Same names, argument meaning and error behaviour as
  /root/reference/src/prover_native.rs:15   pub fn inner_product(A, B) -> Fq12
  /root/reference/src/prover_native.rs:26   pub fn sipp_prove_native(A, B) -> Vec<Fq12>
  /root/reference/src/verifier_native.rs:14 pub fn sipp_verify_native(A, B, proof) -> Result<SIPPStatement>
  /root/reference/src/transcript_native.rs:14-66 Transcript
  /root/reference/src/statements.rs:80-88   SIPPStatement

Values are arkworks canonical little-endian bytes (see include/sipp_b200.h): a G1Affine is 64 bytes, a G2Affine
128 bytes, an Fq12 384 bytes, an Fr 32 bytes.  `A` / `B` may be a list of per-point byte strings (like
`&[G1Affine]`) or one contiguous buffer.  Where the reference panics this module raises (AssertionError for the
`assert_eq!`, SippError otherwise); where it returns `Err` it raises VerificationError.
"""
import ctypes
from dataclasses import dataclass
from typing import List, Sequence, Union

from . import _lib
from ._lib import SippError

G1_BYTES, G2_BYTES, FQ12_BYTES, FR_BYTES = 64, 128, 384, 32
Points = Union[bytes, bytearray, memoryview, Sequence[bytes]]


class VerificationError(Exception):
    """anyhow!("Verification failed")  (verifier_native.rs:83)"""


@dataclass
class SIPPStatement:
    """statements.rs:80-88"""
    A: List[bytes]
    B: List[bytes]
    Z: bytes
    final_A: bytes
    final_B: bytes
    final_Z: bytes

    def to_vec(self) -> List[int]:
        """the u32 public-input vector `SIPPStatement::from_vec` parses (statements.rs:133-170): sipp_statement_to_u32"""
        lib = _lib.load()
        n = len(self.A)
        total = lib.sipp_statement_u32_len(n)
        out = (ctypes.c_uint32 * total)()
        _lib.check(lib.sipp_statement_to_u32(b"".join(self.A), b"".join(self.B), n, self.Z, self.final_A, self.final_B, self.final_Z, out, total))
        return list(out)

    @staticmethod
    def from_vec(n: int, vec: Sequence[int]) -> "SIPPStatement":
        """statements.rs:133-170 (sipp_statement_from_u32), same length assertion"""
        lib = _lib.load()
        arr = (ctypes.c_uint32 * len(vec))(*vec)
        A, B = ctypes.create_string_buffer(max(1, G1_BYTES * n)), ctypes.create_string_buffer(max(1, G2_BYTES * n))
        Z, fa, fb, fz = (ctypes.create_string_buffer(k) for k in (FQ12_BYTES, G1_BYTES, G2_BYTES, FQ12_BYTES))
        rc = lib.sipp_statement_from_u32(n, arr, len(vec), A, B, Z, fa, fb, fz)
        assert rc != _lib.ERR_LENGTH, "assert!(input.len() == total_len)"
        _lib.check(rc)
        return SIPPStatement(A=_split(A.raw[:G1_BYTES * n], G1_BYTES), B=_split(B.raw[:G2_BYTES * n], G2_BYTES), Z=Z.raw, final_A=fa.raw,
                             final_B=fb.raw, final_Z=fz.raw)


# ---- hand-off to the circuit side: statements.rs:90-170 (`SIPPStatement::from_vec`) ---------------------------------------
# The plonky2 verifier circuit takes the statement as one vector of 32-bit limbs (8 little-endian limbs per Fq):
#   A (n x 16) | B (n x 32) | Z (96) | final_A (16) | final_B (32) | final_Z (96)
# G1 / G2 limbs are x | y resp. x.c0 | x.c1 | y.c0 | y.c1 -- byte-identical to the canonical little-endian boundary format.
# An Fq12 is `MyFq12.coeffs` (SURVEY A.2, hypothesis H2 = w-power basis): coeffs[i] = g_i.c0, coeffs[i + 6] = g_i.c1 with
# g_0..g_5 = c0.c0, c1.c0, c0.c1, c1.c1, c0.c2, c1.c2 of the arkworks nested form.
_W_TO_ARK_SLOT = (0, 3, 1, 4, 2, 5)


def fq12_to_myfq12_bytes(f: bytes) -> bytes:
    """ark-serialized Fq12 (384 B) -> the 12 MyFq12 coefficients, 32 little-endian bytes each"""
    assert len(f) == FQ12_BYTES
    fq = [f[32 * i:32 * i + 32] for i in range(12)]
    return b"".join(fq[2 * _W_TO_ARK_SLOT[i]] for i in range(6)) + b"".join(fq[2 * _W_TO_ARK_SLOT[i] + 1] for i in range(6))


def myfq12_bytes_to_fq12(c: bytes) -> bytes:
    assert len(c) == FQ12_BYTES
    co = [c[32 * i:32 * i + 32] for i in range(12)]
    out = [b""] * 12
    for i in range(6):
        out[2 * _W_TO_ARK_SLOT[i]], out[2 * _W_TO_ARK_SLOT[i] + 1] = co[i], co[i + 6]
    return b"".join(out)


def _flat(points: Points, size: int) -> bytes:
    if isinstance(points, (bytes, bytearray, memoryview)):
        b = bytes(points)
    else:
        b = b"".join(bytes(p) for p in points)
    if len(b) % size:
        raise ValueError("buffer length %d is not a multiple of %d" % (len(b), size))
    return b


def _split(b: bytes, size: int) -> List[bytes]:
    return [b[i:i + size] for i in range(0, len(b), size)]


def inner_product(A: Points, B: Points) -> bytes:
    """prod_i e(A_i, B_i)  (prover_native.rs:15-23)"""
    a, b = _flat(A, G1_BYTES), _flat(B, G2_BYTES)
    assert len(a) // G1_BYTES == len(b) // G2_BYTES, "assert_eq!(A.len(), B.len())"  # prover_native.rs:16
    _lib.require_gpu_once()
    out = ctypes.create_string_buffer(FQ12_BYTES)
    _lib.check(_lib.load().sipp_inner_product(a, b, len(a) // G1_BYTES, out))
    return out.raw


def pairing(a: bytes, b: bytes) -> bytes:
    """plonky2_bn254_pairing::pairing::pairing(a, b) as used at verifier_native.rs:80"""
    _lib.require_gpu_once()
    out = ctypes.create_string_buffer(FQ12_BYTES)
    _lib.check(_lib.load().sipp_pairing(bytes(a), bytes(b), out))
    return out.raw


def _offsets(lengths: Sequence[int], n: int):
    """segment sizes -> the count + 1 CSR offsets of sipp_inner_product_batch"""
    offs = [0]
    for length in lengths:
        if length < 0:
            raise ValueError("negative segment length %d" % length)
        offs.append(offs[-1] + int(length))
    if offs[-1] != n:
        raise ValueError("the segment lengths add up to %d, not to the %d pairs" % (offs[-1], n))
    return (ctypes.c_size_t * len(offs))(*offs)


def inner_product_batch(A: Points, B: Points, lengths: Sequence[int]) -> List[bytes]:
    """[inner_product(A[o[j]:o[j+1]], B[o[j]:o[j+1]]) for j < len(lengths)] in one call (sipp_inner_product_batch), o = the running
    sums of `lengths` starting at 0: segment j holds the next lengths[j] pairs, an empty segment gives Fq12::one()"""
    a, b = _flat(A, G1_BYTES), _flat(B, G2_BYTES)
    n = len(a) // G1_BYTES
    assert n == len(b) // G2_BYTES, "assert_eq!(A.len(), B.len())"  # prover_native.rs:16
    offs = _offsets(lengths, n)
    count = len(offs) - 1
    _lib.require_gpu_once()
    out = ctypes.create_string_buffer(max(1, FQ12_BYTES * count))
    _lib.check(_lib.load().sipp_inner_product_batch(a, n, b, n, offs, count, out))
    return _split(out.raw[:FQ12_BYTES * count], FQ12_BYTES)


def pairing_batch(a: Points, b: Points) -> List[bytes]:
    """[pairing(a_j, b_j) for j] in one call (sipp_pairing_batch; verifier_native.rs:80 per pair)"""
    pa, pb = _flat(a, G1_BYTES), _flat(b, G2_BYTES)
    count = len(pa) // G1_BYTES
    assert count == len(pb) // G2_BYTES, "assert_eq!(A.len(), B.len())"
    _lib.require_gpu_once()
    out = ctypes.create_string_buffer(max(1, FQ12_BYTES * count))
    _lib.check(_lib.load().sipp_pairing_batch(pa, pb, count, out))
    return _split(out.raw[:FQ12_BYTES * count], FQ12_BYTES)


def inner_product_batch_device(dA: int, dB: int, n: int, lengths: Sequence[int], d_out: int) -> None:
    """inner_product_batch on DEVICE buffers (integer pointers, e.g. tensor.data_ptr()): dA n x 64 B, dB n x 128 B, d_out
    len(lengths) x 384 B, boundary format (sipp_inner_product_batch_device)"""
    offs = _offsets(lengths, n)
    _lib.require_gpu_once()
    _lib.check(_lib.load().sipp_inner_product_batch_device(dA, dB, n, offs, len(offs) - 1, d_out))


def sipp_prove_native(A: Points, B: Points) -> List[bytes]:
    """prover_native.rs:26-80; returns the proof as a list of 2 log2(n) + 1 Fq12 byte strings."""
    a, b = _flat(A, G1_BYTES), _flat(B, G2_BYTES)
    na, nb = len(a) // G1_BYTES, len(b) // G2_BYTES
    assert na == nb, "assert_eq!(A.len(), B.len())"  # prover_native.rs:27
    _lib.require_gpu_once()
    lib = _lib.load()
    plen = lib.sipp_proof_len(na)
    if plen == 0:
        raise SippError(_lib.ERR_ARG, "n must be a non-zero power of two")
    proof = ctypes.create_string_buffer(FQ12_BYTES * plen)
    _lib.check(lib.sipp_prove_native(a, na, b, nb, proof))
    return _split(proof.raw, FQ12_BYTES)


def sipp_prove_native_batch(A: Points, B: Points, n: int) -> List[List[bytes]]:
    """`count` independent instances of `n` pairs each, proved in lock-step on the device (one Fiat-Shamir chain per instance
    on the GPU): proofs[j] == sipp_prove_native(A[j*n:(j+1)*n], B[j*n:(j+1)*n])  (prover_native.rs:26-80 per instance)."""
    a, b = _flat(A, G1_BYTES), _flat(B, G2_BYTES)
    na, nb = len(a) // G1_BYTES, len(b) // G2_BYTES
    assert na == nb, "assert_eq!(A.len(), B.len())"  # prover_native.rs:27
    if n <= 0 or na % n:
        raise ValueError("the number of pairs (%d) is not a multiple of the instance size %d" % (na, n))
    count = na // n
    _lib.require_gpu_once()
    lib = _lib.load()
    plen = lib.sipp_proof_len(n)
    if plen == 0:
        raise SippError(_lib.ERR_ARG, "n must be a non-zero power of two")
    proofs = ctypes.create_string_buffer(FQ12_BYTES * plen * count)
    _lib.check(lib.sipp_prove_native_batch(a, b, n, count, proofs))
    raw = proofs.raw
    return [_split(raw[j * plen * FQ12_BYTES:(j + 1) * plen * FQ12_BYTES], FQ12_BYTES) for j in range(count)]


def _ragged_offsets(lengths: Sequence[int], n: int):
    """instance sizes -> the count + 1 CSR offsets of sipp_prove_native_batch_ragged; every size a non-zero power of two"""
    for length in lengths:
        if int(length) <= 0 or int(length) & (int(length) - 1):
            raise ValueError("instance size %d is not a non-zero power of two" % length)
    return _offsets(lengths, n)


def sipp_prove_native_batch_ragged(A: Points, B: Points, lengths: Sequence[int]) -> List[List[bytes]]:
    """Independent instances of different sizes, proved in lock-step on the device (sipp_prove_native_batch_ragged): instance j is
    the next lengths[j] pairs (a power of two) and proofs[j] == sipp_prove_native(A[o[j]:o[j+1]], B[o[j]:o[j+1]]), o = the running
    sums of `lengths` starting at 0.  A bad point or a zero challenge fails the whole call (SippError) and returns no proof.

    The registration of A and B in each instance's transcript is a device chain of 8 n_j Poseidon permutations, and the longest
    instance bounds it: an instance far larger than the rest is better proved on its own with sipp_prove_native."""
    a, b = _flat(A, G1_BYTES), _flat(B, G2_BYTES)
    n = len(a) // G1_BYTES
    assert n == len(b) // G2_BYTES, "assert_eq!(A.len(), B.len())"  # prover_native.rs:27
    offs = _ragged_offsets(lengths, n)
    count = len(offs) - 1
    if count == 0:
        raise ValueError("no instances")
    _lib.require_gpu_once()
    lib = _lib.load()
    plens = [lib.sipp_proof_len(int(length)) for length in lengths]
    proofs = ctypes.create_string_buffer(FQ12_BYTES * sum(plens))
    _lib.check(lib.sipp_prove_native_batch_ragged(a, n, b, n, offs, count, proofs))
    raw, out, pos = proofs.raw, [], 0
    for plen in plens:
        out.append(_split(raw[pos:pos + plen * FQ12_BYTES], FQ12_BYTES))
        pos += plen * FQ12_BYTES
    return out


def sipp_prove_native_batch_ragged_device(dA: int, dB: int, n: int, lengths: Sequence[int], d_proofs: int) -> None:
    """sipp_prove_native_batch_ragged on DEVICE buffers (integer pointers, e.g. tensor.data_ptr()): dA n x 64 B, dB n x 128 B,
    d_proofs sum_j (2 log2 lengths[j] + 1) x 384 B, boundary format; instance j's proof follows those of instances 0 .. j - 1"""
    offs = _ragged_offsets(lengths, n)
    _lib.require_gpu_once()
    _lib.check(_lib.load().sipp_prove_native_batch_ragged_device(dA, dB, n, offs, len(offs) - 1, d_proofs))


def sipp_verify_native_batch(A: Points, B: Points, n: int, proofs: Sequence[Sequence[bytes]]) -> List[Union[SIPPStatement, VerificationError]]:
    """`count` independent verifications in lock-step (verifier_native.rs:14-85 per instance).  Returns, per instance, the
    SIPPStatement (Ok) or a VerificationError instance (Err) -- a failed instance does not abort the others."""
    a, b = _flat(A, G1_BYTES), _flat(B, G2_BYTES)
    na, nb = len(a) // G1_BYTES, len(b) // G2_BYTES
    assert na == nb, "assert_eq!(A.len(), B.len())"
    if n <= 0 or na % n or na // n != len(proofs):
        raise ValueError("%d pairs / instance size %d does not match %d proofs" % (na, n, len(proofs)))
    count = na // n
    plen = len(proofs[0])
    if any(len(p) != plen for p in proofs):
        raise ValueError("all proofs of a batch must have the same length")
    p = b"".join(_flat(pr, FQ12_BYTES) for pr in proofs)
    _lib.require_gpu_once()
    res = (ctypes.c_int * count)()
    fa, fb, fz = (ctypes.create_string_buffer(s * count) for s in (G1_BYTES, G2_BYTES, FQ12_BYTES))
    _lib.check(_lib.load().sipp_verify_native_batch(a, b, n, count, p, plen, res, fa, fb, fz))
    out = []
    for j in range(count):
        if res[j] == _lib.ERR_VERIFY:
            out.append(VerificationError("Verification failed"))
        else:
            out.append(SIPPStatement(A=_split(a[G1_BYTES * n * j:G1_BYTES * n * (j + 1)], G1_BYTES),
                                     B=_split(b[G2_BYTES * n * j:G2_BYTES * n * (j + 1)], G2_BYTES), Z=bytes(proofs[j][-1]),
                                     final_A=fa.raw[G1_BYTES * j:G1_BYTES * (j + 1)], final_B=fb.raw[G2_BYTES * j:G2_BYTES * (j + 1)],
                                     final_Z=fz.raw[FQ12_BYTES * j:FQ12_BYTES * (j + 1)]))
    return out


def sipp_verify_native_batch_ragged(A: Points, B: Points, lengths: Sequence[int],
                                    proofs: Sequence[Sequence[bytes]]) -> List[Union[SIPPStatement, VerificationError, SippError]]:
    """Independent verifications of instances of different sizes in lock-step (sipp_verify_native_batch_ragged): instance j is the
    next lengths[j] pairs (a power of two) with proof proofs[j] (a list of Fq12 byte strings or one buffer, read from its end), as
    sipp_prove_native_batch_ragged returns them.  Returns, per instance, what sipp_verify_native gives on it: the SIPPStatement (Ok),
    a VerificationError instance (Err), or a SippError instance with code ERR_ENCODING for a proof with a coordinate >= p -- a
    failed instance does not abort the others.  A bad point, a zero challenge or a short proof fails the whole call (SippError).

    As for the prover, the registration of A and B is a device chain of 8 n_j Poseidon permutations per instance and the longest
    instance bounds it: an instance far larger than the rest is better verified on its own with sipp_verify_native."""
    a, b = _flat(A, G1_BYTES), _flat(B, G2_BYTES)
    n = len(a) // G1_BYTES
    assert n == len(b) // G2_BYTES, "assert_eq!(A.len(), B.len())"
    offs = _ragged_offsets(lengths, n)
    count = len(offs) - 1
    if count == 0:
        raise ValueError("no instances")
    if len(proofs) != count:
        raise ValueError("%d instances but %d proofs" % (count, len(proofs)))
    flat = [_flat(p, FQ12_BYTES) for p in proofs]
    poffs = [0]
    for p in flat:
        poffs.append(poffs[-1] + len(p) // FQ12_BYTES)
    _lib.require_gpu_once()
    res = (ctypes.c_int * count)()
    fa, fb, fz = (ctypes.create_string_buffer(s * count) for s in (G1_BYTES, G2_BYTES, FQ12_BYTES))
    _lib.check(_lib.load().sipp_verify_native_batch_ragged(a, n, b, n, offs, count, b"".join(flat), (ctypes.c_size_t * len(poffs))(*poffs), res,
                                                           fa, fb, fz))
    out = []
    for j in range(count):
        if res[j] == _lib.OK:
            out.append(SIPPStatement(A=_split(a[G1_BYTES * offs[j]:G1_BYTES * offs[j + 1]], G1_BYTES),
                                     B=_split(b[G2_BYTES * offs[j]:G2_BYTES * offs[j + 1]], G2_BYTES), Z=flat[j][-FQ12_BYTES:],
                                     final_A=fa.raw[G1_BYTES * j:G1_BYTES * (j + 1)], final_B=fb.raw[G2_BYTES * j:G2_BYTES * (j + 1)],
                                     final_Z=fz.raw[FQ12_BYTES * j:FQ12_BYTES * (j + 1)]))
        elif res[j] == _lib.ERR_VERIFY:
            out.append(VerificationError("Verification failed"))
        elif res[j] == _lib.ERR_ENCODING:
            out.append(SippError(_lib.ERR_ENCODING, "instance %d: proof coordinate >= p" % j))
        else:
            out.append(SippError(res[j], "instance %d: unexpected result" % j))
    return out


def sipp_verify_native(A: Points, B: Points, proof: Sequence[bytes]) -> SIPPStatement:
    """verifier_native.rs:14-85; returns the SIPPStatement or raises VerificationError."""
    a, b = _flat(A, G1_BYTES), _flat(B, G2_BYTES)
    p = _flat(proof, FQ12_BYTES)
    na, nb = len(a) // G1_BYTES, len(b) // G2_BYTES
    _lib.require_gpu_once()
    fa, fb, fz = (ctypes.create_string_buffer(s) for s in (G1_BYTES, G2_BYTES, FQ12_BYTES))
    rc = _lib.load().sipp_verify_native(a, na, b, nb, p, len(p) // FQ12_BYTES, fa, fb, fz)
    if rc == _lib.ERR_VERIFY:
        raise VerificationError("Verification failed")
    _lib.check(rc)
    return SIPPStatement(A=_split(a, G1_BYTES), B=_split(b, G2_BYTES), Z=p[-FQ12_BYTES:], final_A=fa.raw, final_B=fb.raw, final_Z=fz.raw)


class Transcript:
    """transcript_native.rs:14-66 (host code: usable without a GPU)."""

    def __init__(self):
        self._t = _lib.TranscriptState()
        _lib.load().sipp_transcript_new(ctypes.byref(self._t))

    @property
    def state(self) -> List[int]:
        return list(self._t.state)

    def append(self, message: Sequence[int]) -> None:
        arr = (ctypes.c_uint64 * max(1, len(message)))(*message)
        _lib.load().sipp_transcript_append(ctypes.byref(self._t), arr, len(message))

    def append_fq12(self, x: bytes) -> None:
        assert len(x) == FQ12_BYTES
        _lib.load().sipp_transcript_append_fq12(ctypes.byref(self._t), bytes(x))

    def append_g1(self, p: bytes) -> None:
        assert len(p) == G1_BYTES
        _lib.load().sipp_transcript_append_g1(ctypes.byref(self._t), bytes(p))

    def append_g2(self, x: bytes) -> None:
        assert len(x) == G2_BYTES
        _lib.load().sipp_transcript_append_g2(ctypes.byref(self._t), bytes(x))

    def get_challenge(self) -> bytes:
        out = ctypes.create_string_buffer(FR_BYTES)
        _lib.load().sipp_transcript_get_challenge(ctypes.byref(self._t), out)
        return out.raw


class ProverContext:
    """Round-granular access to the device-resident prover state (sipp_ctx_*): what a host that keeps its own
    transcript calls between challenges (prover_native.rs:29, :48-49, :60-74)."""

    def __init__(self, A: Points = None, B: Points = None, device_ptrs=None, n=None):
        _lib.require_gpu_once()
        self._h = ctypes.c_void_p()
        lib = _lib.load()
        if device_ptrs is not None:
            _lib.check(lib.sipp_ctx_create_from_device(device_ptrs[0], device_ptrs[1], n, ctypes.byref(self._h)))
        else:
            a, b = _flat(A, G1_BYTES), _flat(B, G2_BYTES)
            assert len(a) // G1_BYTES == len(b) // G2_BYTES
            _lib.check(lib.sipp_ctx_create(a, b, len(a) // G1_BYTES, ctypes.byref(self._h)))

    def __len__(self):
        return _lib.load().sipp_ctx_len(self._h)

    def inner_product(self) -> bytes:
        out = ctypes.create_string_buffer(FQ12_BYTES)
        _lib.check(_lib.load().sipp_ctx_inner_product(self._h, out))
        return out.raw

    def cross_products(self):
        zl, zr = ctypes.create_string_buffer(FQ12_BYTES), ctypes.create_string_buffer(FQ12_BYTES)
        _lib.check(_lib.load().sipp_ctx_cross_products(self._h, zl, zr))
        return zl.raw, zr.raw

    def fold(self, x: bytes, x_inv: bytes) -> None:
        _lib.check(_lib.load().sipp_ctx_fold(self._h, bytes(x), bytes(x_inv)))

    def set_stages(self, on: bool = True) -> None:
        """opt in to the pairing-matrix stages for inner_product / cross_products / fold (sipp_ctx_set_stages): same values,
        shorter rounds; read() is refused once the tail stage has begun"""
        _lib.check(_lib.load().sipp_ctx_set_stages(self._h, 1 if on else 0))

    def read(self):
        n = len(self)
        a, b = ctypes.create_string_buffer(G1_BYTES * n), ctypes.create_string_buffer(G2_BYTES * n)
        _lib.check(_lib.load().sipp_ctx_read(self._h, a, b))
        return a.raw, b.raw

    def prove(self, A: Points, B: Points) -> List[bytes]:
        a, b = _flat(A, G1_BYTES), _flat(B, G2_BYTES)
        lib = _lib.load()
        plen = lib.sipp_proof_len(len(self))
        proof = ctypes.create_string_buffer(FQ12_BYTES * plen)
        _lib.check(lib.sipp_ctx_prove(self._h, a, b, proof))
        return _split(proof.raw, FQ12_BYTES)

    def partial_products(self, which: int, d_out: int, stream: int = 0) -> None:
        _lib.check(_lib.load().sipp_ctx_partial_products(self._h, which, d_out, stream))

    def close(self):
        if self._h:
            _lib.load().sipp_ctx_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def combine_partials(d_partials: int, count: int, nprod: int, stream: int = 0) -> List[bytes]:
    out = ctypes.create_string_buffer(FQ12_BYTES * nprod)
    _lib.check(_lib.load().sipp_combine_partials(d_partials, count, nprod, out, stream))
    return _split(out.raw, FQ12_BYTES)


def fr_inverse(x: bytes) -> bytes:
    out = ctypes.create_string_buffer(FR_BYTES)
    _lib.check(_lib.load().sipp_fr_inverse(bytes(x), out))
    return out.raw


# ---- input producers of the BLS-aggregation demo (bin/bls_aggregation.rs:95-117) ---------------------------------------------
def g1_generator_mul_batch(scalars: Points) -> List[bytes]:
    """public_keys[i] = (G1Affine::generator() * sk_i).into()   (bls_aggregation.rs:96-99)"""
    k = _flat(scalars, FR_BYTES)
    _lib.require_gpu_once()
    out = ctypes.create_string_buffer(G1_BYTES * (len(k) // FR_BYTES))
    _lib.check(_lib.load().sipp_g1_generator_mul_batch(k, len(k) // FR_BYTES, out))
    return _split(out.raw, G1_BYTES)


def g2_mul_batch(points: Points, scalars: Points) -> List[bytes]:
    """signatures[i] = (m_i * sk_i).into()   (bls_aggregation.rs:105-109); a single point multiplies every scalar"""
    p, k = _flat(points, G2_BYTES), _flat(scalars, FR_BYTES)
    _lib.require_gpu_once()
    count = len(k) // FR_BYTES
    out = ctypes.create_string_buffer(G2_BYTES * count)
    _lib.check(_lib.load().sipp_g2_mul_batch(p, len(p) // G2_BYTES, k, count, out))
    return _split(out.raw, G2_BYTES)


def g2_sum(points: Points) -> bytes:
    """signatures.iter().fold(G2Projective::zero(), |acc, &s| acc + s).into()   (bls_aggregation.rs:110-113)"""
    p = _flat(points, G2_BYTES)
    _lib.require_gpu_once()
    out = ctypes.create_string_buffer(G2_BYTES)
    _lib.check(_lib.load().sipp_g2_sum(p, len(p) // G2_BYTES, out))
    return out.raw


def g1_neg_generator() -> bytes:
    """-G1Affine::generator()   (bls_aggregation.rs:116)"""
    out = ctypes.create_string_buffer(G1_BYTES)
    _lib.check(_lib.load().sipp_g1_neg_generator(out))
    return out.raw


def seeded_inputs(seed: int, n: int):
    """A_i = [a_i]G1, B_i = [b_i]G2 with the documented SplitMix64 scalar stream, generated on the GPU."""
    _lib.require_gpu_once()
    a, b = ctypes.create_string_buffer(G1_BYTES * n), ctypes.create_string_buffer(G2_BYTES * n)
    _lib.check(_lib.load().sipp_seeded_inputs(seed, n, a, b))
    return a.raw, b.raw


def stats(reset=False) -> dict:
    s = _lib.Stats()
    _lib.check(_lib.load().sipp_get_stats(ctypes.byref(s)))
    if reset:
        _lib.load().sipp_reset_stats()
    return {k: getattr(s, k) for k, _ in _lib.Stats._fields_}


def set_option(option: int, value: int) -> None:
    _lib.check(_lib.load().sipp_set_option(option, value))
