"""ctypes loader for libsipp_b200.so (the C ABI declared in include/sipp_b200.h).

The library is built in-tree by `make -C sipp_b200/csrc` (see __graft_entry__.build).  There is no fallback: if
the shared object is missing, or no CUDA device is usable, every compute call raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SIPP_LIB") or os.path.join(_HERE, "libsipp_b200.so")  # SIPP_LIB: A/B builds of the same ABI

OK, ERR_CUDA, ERR_ARG, ERR_LENGTH, ERR_ZERO_CHALLENGE, ERR_SHORT_PROOF, ERR_ENCODING, ERR_VERIFY, ERR_COMM = 0, -1, -2, -3, -4, -5, -6, -7, -8
OPT_FE_NORMALISATION, OPT_FQ12_ORDER, OPT_PROFILE, OPT_PIPELINE, OPT_WIDE_LINES_MAX, OPT_FE_ENGINE, OPT_WIDE_FOLD_MAX, OPT_WIDE_ACCUM_MAX = 1, 2, 3, 4, 5, 6, 7, 8
OPT_BATCH_KPG_MAX, OPT_FOLD_STRAUS, OPT_BATCH_STREAMS, OPT_BATCH_QLINES, OPT_VALIDATE_POINTS, OPT_MATRIX_TAIL, OPT_MATRIX_BLOCK_N, OPT_MATRIX_BLOCK_R, OPT_MATRIX_FIRST = 9, 10, 11, 12, 13, 14, 15, 16, 17
OPT_PRODUCT_CHUNK_PAIRS = 18


class SippError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libsipp_b200 error %d: %s" % (code, msg))
        self.code = code


class Stats(ctypes.Structure):
    _fields_ = [("launches", ctypes.c_uint64), ("miller_pairs", ctypes.c_uint64), ("miller_launches", ctypes.c_uint64),
                ("miller_ms", ctypes.c_double), ("reduce_fe_ms", ctypes.c_double), ("fold_ms", ctypes.c_double),
                ("fold_points", ctypes.c_uint64), ("transcript_ms", ctypes.c_double), ("other_ms", ctypes.c_double)]


class TranscriptState(ctypes.Structure):
    _fields_ = [("state", ctypes.c_uint64 * 4)]


ALLGATHER_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t)
BROADCAST_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int)
SHARD_XS_BYTES = 72


class ShardBackend(ctypes.Structure):
    """sipp_shard_backend (include/sipp_b200.h): the compute / exchange side of the sharded protocol loop"""
    LEN_FN = ctypes.CFUNCTYPE(ctypes.c_size_t, ctypes.c_void_p)
    PRODUCTS_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_int)
    COMBINE_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p)
    BROADCAST_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p)
    FOLD_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p)
    COLLAPSE_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p)
    _fields_ = [("user", ctypes.c_void_p), ("rank", ctypes.c_int), ("world", ctypes.c_int), ("local_len", LEN_FN), ("products", PRODUCTS_FN),
                ("combine", COMBINE_FN), ("broadcast", BROADCAST_FN), ("fold", FOLD_FN), ("collapse", COLLAPSE_FN)]


_lib = None


def load():
    """dlopen the C-ABI library; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SippError(ERR_CUDA, "%s not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                  "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, sz, u8p, i = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_int
    lib.sipp_last_error.restype = ctypes.c_char_p
    lib.sipp_ctx_create.argtypes = [u8p, u8p, sz, ctypes.POINTER(vp)]
    lib.sipp_poseidon_ns_per_permutation.argtypes = [ctypes.c_long]
    lib.sipp_poseidon_ns_per_permutation.restype = ctypes.c_double
    lib.sipp_ctx_create_from_device.argtypes = [vp, vp, sz, ctypes.POINTER(vp)]
    lib.sipp_ctx_destroy.argtypes = [vp]
    lib.sipp_ctx_len.argtypes = [vp]
    lib.sipp_ctx_len.restype = sz
    lib.sipp_ctx_inner_product.argtypes = [vp, u8p]
    lib.sipp_ctx_cross_products.argtypes = [vp, u8p, u8p]
    lib.sipp_ctx_fold.argtypes = [vp, u8p, u8p]
    lib.sipp_ctx_read.argtypes = [vp, u8p, u8p]
    lib.sipp_ctx_set_stages.argtypes = [vp, ctypes.c_int]
    lib.sipp_ctx_partial_products.argtypes = [vp, i, vp, vp]
    lib.sipp_combine_partials.argtypes = [vp, i, i, u8p, vp]
    lib.sipp_pairing.argtypes = [u8p, u8p, u8p]
    lib.sipp_inner_product.argtypes = [u8p, u8p, sz, u8p]
    lib.sipp_fr_inverse.argtypes = [u8p, u8p]
    lib.sipp_gt_fold.argtypes = [u8p, u8p, u8p, u8p, u8p, u8p]
    szp = ctypes.POINTER(ctypes.c_size_t)
    lib.sipp_inner_product_batch.argtypes = [u8p, sz, u8p, sz, szp, sz, u8p]
    lib.sipp_inner_product_batch_device.argtypes = [vp, vp, sz, szp, sz, vp]
    lib.sipp_pairing_batch.argtypes = [u8p, u8p, sz, u8p]
    lib.sipp_test_product_plan.argtypes = [szp, sz, i, sz, szp, sz, ctypes.POINTER(ctypes.c_int)]
    lib.sipp_test_product_plan.restype = ctypes.c_long
    lib.sipp_test_ragged_schedule.argtypes = [szp, sz, ctypes.POINTER(ctypes.c_longlong), sz]
    lib.sipp_test_ragged_schedule.restype = ctypes.c_long
    lib.sipp_transcript_new.argtypes = [ctypes.POINTER(TranscriptState)]
    lib.sipp_transcript_new.restype = None
    lib.sipp_transcript_append.argtypes = [ctypes.POINTER(TranscriptState), ctypes.POINTER(ctypes.c_uint64), sz]
    lib.sipp_transcript_append.restype = None
    for name in ("sipp_transcript_append_fq12", "sipp_transcript_append_g1", "sipp_transcript_append_g2"):
        getattr(lib, name).argtypes = [ctypes.POINTER(TranscriptState), u8p]
        getattr(lib, name).restype = None
    lib.sipp_transcript_get_challenge.argtypes = [ctypes.POINTER(TranscriptState), u8p]
    lib.sipp_transcript_get_challenge.restype = None
    lib.sipp_transcript_append_pairs.argtypes = [ctypes.POINTER(TranscriptState), u8p, u8p, sz]
    lib.sipp_transcript_append_pairs.restype = None
    lib.sipp_poseidon_permute.argtypes = [ctypes.POINTER(ctypes.c_uint64)]
    lib.sipp_poseidon_permute.restype = None
    lib.sipp_prove_native.argtypes = [u8p, sz, u8p, sz, u8p]
    lib.sipp_proof_len.argtypes = [sz]
    lib.sipp_proof_len.restype = sz
    lib.sipp_ctx_prove.argtypes = [vp, u8p, u8p, u8p]
    lib.sipp_verify_native.argtypes = [u8p, sz, u8p, sz, u8p, sz, u8p, u8p, u8p]
    lib.sipp_seeded_inputs_device.argtypes = [ctypes.c_uint64, sz, vp, vp]
    lib.sipp_seeded_inputs.argtypes = [ctypes.c_uint64, sz, u8p, u8p]
    lib.sipp_get_stats.argtypes = [ctypes.POINTER(Stats)]
    lib.sipp_test_fq_op.argtypes = [i, u8p, u8p, u8p, sz]
    lib.sipp_test_fq12_op.argtypes = [i, u8p, u8p, u8p, sz]
    lib.sipp_prove_native_batch.argtypes = [u8p, u8p, sz, sz, u8p]
    lib.sipp_prove_native_batch_device.argtypes = [vp, vp, sz, sz, vp]
    lib.sipp_prove_native_batch_ragged.argtypes = [u8p, sz, u8p, sz, szp, sz, u8p]
    lib.sipp_prove_native_batch_ragged_device.argtypes = [vp, vp, sz, szp, sz, vp]
    lib.sipp_prove_native_statement.argtypes = [u8p, sz, u8p, sz, u8p, u8p, u8p, u8p]
    lib.sipp_prove_native_batch_statement.argtypes = [u8p, u8p, sz, sz, u8p, u8p, u8p, u8p]
    lib.sipp_prove_native_batch_statement_device.argtypes = [vp, vp, sz, sz, vp, vp, vp, vp]
    lib.sipp_prove_native_batch_ragged_statement.argtypes = [u8p, sz, u8p, sz, szp, sz, u8p, u8p, u8p, u8p]
    lib.sipp_prove_native_batch_ragged_statement_device.argtypes = [vp, vp, sz, szp, sz, vp, vp, vp, vp]
    lib.sipp_verify_native_batch.argtypes = [u8p, u8p, sz, sz, u8p, sz, ctypes.POINTER(ctypes.c_int), u8p, u8p, u8p]
    lib.sipp_verify_native_batch_ragged.argtypes = [u8p, sz, u8p, sz, szp, sz, u8p, szp, ctypes.POINTER(ctypes.c_int), u8p, u8p, u8p]
    lib.sipp_verify_native_batch_device.argtypes = [vp, vp, sz, sz, vp, sz, vp, vp, vp, vp]
    lib.sipp_verify_native_batch_ragged_device.argtypes = [vp, vp, sz, szp, sz, vp, szp, vp, vp, vp, vp]
    lib.sipp_test_poseidon_device.argtypes = [ctypes.POINTER(ctypes.c_uint64), sz]
    lib.sipp_test_transcript_round_device.argtypes = [ctypes.POINTER(ctypes.c_uint64), u8p, i, sz, u8p, ctypes.POINTER(ctypes.c_uint32)]
    lib.sipp_test_fold_plan.argtypes = [u8p, u8p, ctypes.POINTER(ctypes.c_uint32), sz]
    u32p = ctypes.POINTER(ctypes.c_uint32)
    lib.sipp_test_fold_plan_device.argtypes = [u8p, u8p, sz, u32p]
    lib.sipp_test_fold_batch.argtypes = [u8p, u8p, sz, sz, u8p, u8p, i, u8p, u8p]
    lib.sipp_statement_u32_len.argtypes = [sz]
    lib.sipp_statement_u32_len.restype = sz
    lib.sipp_statement_to_u32.argtypes = [u8p, u8p, sz, u8p, u8p, u8p, u8p, u32p, sz]
    lib.sipp_statement_from_u32.argtypes = [sz, u32p, sz, u8p, u8p, u8p, u8p, u8p, u8p]
    lib.sipp_g1_generator_mul_batch.argtypes = [u8p, sz, u8p]
    lib.sipp_g1_generator_mul_batch_device.argtypes = [vp, sz, vp]
    lib.sipp_g2_mul_batch.argtypes = [u8p, sz, u8p, sz, u8p]
    lib.sipp_g2_mul_batch_device.argtypes = [vp, sz, vp, sz, vp]
    lib.sipp_g2_sum.argtypes = [u8p, sz, u8p]
    lib.sipp_g2_sum_device.argtypes = [vp, sz, vp]
    lib.sipp_g1_neg_generator.argtypes = [u8p]
    for name in ("sipp_g1_msm_batch", "sipp_g2_msm_batch"):
        getattr(lib, name).argtypes = [u8p, u8p, sz, szp, sz, u8p]
    for name in ("sipp_g1_msm_batch_device", "sipp_g2_msm_batch_device"):
        getattr(lib, name).argtypes = [vp, vp, sz, szp, sz, vp]
    lib.sipp_test_msm_plan.argtypes = [szp, sz, ctypes.POINTER(ctypes.c_int), sz]
    lib.sipp_test_msm_plan.restype = ctypes.c_long
    lib.sipp_test_msm_batch_device.argtypes = [i, i, vp, vp, sz, szp, sz, vp]
    lib.sipp_gt_msm_batch.argtypes = [u8p, u8p, sz, szp, sz, u8p]
    lib.sipp_gt_msm_batch_device.argtypes = [vp, vp, sz, szp, sz, vp]
    lib.sipp_test_gt_msm_plan.argtypes = [szp, sz, ctypes.POINTER(ctypes.c_int), sz]
    lib.sipp_test_gt_msm_plan.restype = ctypes.c_long
    lib.sipp_test_gt_msm_batch_device.argtypes = [i, vp, vp, sz, szp, sz, vp]
    lib.sipp_comm_get_unique_id.argtypes = [u8p]
    lib.sipp_comm_init.argtypes = [u8p, i, i]
    lib.sipp_comm_init_host.argtypes = [i, i, ALLGATHER_FN, BROADCAST_FN, vp]
    lib.sipp_prove_native_sharded.argtypes = [u8p, u8p, sz, u8p, u8p, u8p]
    lib.sipp_prove_native_sharded_device.argtypes = [vp, vp, sz, u8p, u8p, u8p]
    lib.sipp_prove_native_sharded_backend.argtypes = [ctypes.POINTER(ShardBackend), sz, u8p, u8p, u8p]
    lib.sipp_microbench.argtypes = [i, i, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
    _lib = lib
    return lib


def check(rc):
    if rc != OK:
        raise SippError(rc, load().sipp_last_error().decode("utf-8", "replace"))
    return rc


def require_gpu(device=0):
    """Select the CUDA device; raises SippError if there is none (the product has no CPU path)."""
    check(load().sipp_init(device))


_gpu_ready = False


def require_gpu_once():
    global _gpu_ready
    if not _gpu_ready:
        dev = int(os.environ.get("LOCAL_RANK", "0")) if "SIPP_DEVICE" not in os.environ else int(os.environ["SIPP_DEVICE"])
        require_gpu(dev)
        _gpu_ready = True
