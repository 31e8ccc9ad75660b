"""sipp_b200 -- B200-native (sm_100a) implementation of qope/SIPP's native prover hot path.

The product is the C-ABI shared library `libsipp_b200.so` (include/sipp_b200.h); this package is the thin host
mirror of the reference interface used by the tests and bench.py.  Nothing here computes on the CPU except the
Poseidon transcript, which the reference also keeps on the host.
"""
from .api import (ProverContext, SIPPStatement, Transcript, VerificationError, combine_partials, fr_inverse,  # noqa: F401
                  g1_generator_mul_batch, g1_neg_generator, g2_mul_batch, g2_sum, inner_product, inner_product_batch, inner_product_batch_device,
                  pairing, pairing_batch, seeded_inputs, set_option, sipp_prove_native, sipp_prove_native_batch,
                  sipp_prove_native_batch_ragged, sipp_prove_native_batch_ragged_device, sipp_verify_native, sipp_verify_native_batch,
                  sipp_verify_native_batch_ragged, stats)
from ._lib import SippError  # noqa: F401
