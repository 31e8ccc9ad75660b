"""The CPU oracle under the four conventions that cannot be settled offline (DESIGN.md §2): H1, the final-exponentiation
normalisation (bit oracle.FE_ARK), and H2, the order in which the transcript absorbs an Fq12 (bit oracle.FQ12_NESTED).  The GPU
tests of every convention (tests/test_gpu_options.py) take the oracle as their reference, so here it is pinned to the
independent pure-Python model (tests/golden/sipp_model.py) byte for byte, and its verifier must accept a proof under exactly
the convention the proof was made with.  CPU only."""
import os
import sys

import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import sipp_model as model  # noqa: E402

CONVENTIONS = (0, 1, 2, 3)


def _model_args(opts, oracle):
    return ("ark" if opts & oracle.FE_ARK else "exact"), ("nested" if opts & oracle.FQ12_NESTED else "wbasis")


def _inputs(seed, n):
    """model points and their raw boundary bytes, serialised as tests/golden/gen_golden.py does"""
    A, B = model.seeded_inputs(seed, n)
    return A, B, b"".join(model.g1_raw(p) for p in A), b"".join(model.g2_raw(q) for q in B)


@pytest.mark.parametrize("n,opts", [(2, o) for o in CONVENTIONS] + [(4, o) for o in CONVENTIONS] + [(8, 3)])
def test_oracle_proof_equals_model(oracle, n, opts):
    A, B, a, b = _inputs(300 + n, n)
    norm, order = _model_args(opts, oracle)
    want = model.proof_bytes(model.sipp_prove_native(A, B, normalisation=norm, order=order))
    assert oracle.sipp_prove(a, b, opts) == want
    assert oracle.seeded_inputs(300 + n, n) == (a, b)   # the GPU tests build their inputs with the oracle's generator


def test_oracle_conventions_differ_and_verify_only_their_own(oracle):
    """n = 8: the four proofs of one input are pairwise different, and oracle.sipp_verify accepts exactly on the diagonal"""
    a, b = oracle.seeded_inputs(308, 8)
    proofs = {o: oracle.sipp_prove(a, b, o, threads=4) for o in CONVENTIONS}
    assert len(set(proofs.values())) == len(CONVENTIONS)
    for made in CONVENTIONS:
        for checked in CONVENTIONS:
            ok, _ = oracle.sipp_verify(a, b, proofs[made], checked, threads=4)
            assert ok == (made == checked), (made, checked)
