"""SEAL-named ABI layer (include/b200_sealc.h) on the CPU emulation build: FFI call sequences of seal_fhe replayed
against our library and the reference, every word / HRESULT compared."""
import pytest

import sealc_checks as sc
from params import PARAMS
from sealc_driver import Sealc


@pytest.fixture(scope="module")
def S(emu_lib):
    return Sealc(emu_lib.lib)


def test_simple_multiply_ffi_sequence(S, ref):
    sc.simple_multiply_sequence(S, *PARAMS["n4096"])


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_evaluator_surface(S, ref_or_none, name):
    sc.evaluator_surface(S, *PARAMS[name])


def test_error_codes(S, ref_or_none):
    sc.error_codes(S, ref_or_none, *PARAMS["n4096"])


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_seeded_encryption_matches_reference(S, ref, name):
    sc.seeded_encryption_parity(S, *PARAMS[name])


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_keygen_and_encryptor_interoperate_with_reference(S, ref, name):
    sc.keygen_interop(S, *PARAMS[name])


def test_chi_sq_dag_small(S, ref):
    sc.chi_sq_dag(S, *PARAMS["n8192"], evaluations=1)


@pytest.mark.parametrize("name", ["n8192"])
def test_batch_encoder(S, ref_or_none, name):
    sc.batch_encoder_parity(S, *PARAMS[name])


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_wire_format(S, ref, name):
    sc.wire_format(S, *PARAMS[name])


def test_polynomial_array(S, ref):
    sc.polynomial_array_parity(S, *PARAMS["n4096"])


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_encryption_components(S, ref, name):
    sc.encryption_components_parity(S, *PARAMS[name])


def test_leftover_entry_points(S, ref):
    sc.leftovers_parity(S, *PARAMS["n4096"])


def test_seal_fhe_golden_fixture(S, ref):
    import os
    sc.seal_fhe_golden_fixture(S, os.path.join(os.path.dirname(__file__), "golden", "seal_fhe_data"))


@pytest.mark.parametrize("n,moduli,t", [(1024, [0x7e00001], 1 << 8), (2048, [0x3fffffff000001], 65537)])
def test_single_prime_chain(S, ref, n, moduli, t):
    sc.single_prime_context(S, n, moduli, t)


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_whole_chain_and_large_sizes(S, ref, name):
    sc.deep_chain_parity(S, *PARAMS[name])


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_misuse_hresults(S, ref, name):
    sc.misuse_hresults(S, *PARAMS[name])


def test_context_validation_sweep(S, ref_or_none):
    sc.context_validation_sweep(S)


def test_concurrent_evaluator_calls(S, ref):
    sc.concurrent_evaluator_calls(S, *PARAMS["n4096"], threads=6, rounds=3)
    sc.concurrent_evaluator_calls(S, *PARAMS["n8192"], threads=4, rounds=2)  # batching plain modulus: rotations too


def test_combined_calls_isolation(S, ref):
    sc.combined_calls_isolation(S, *PARAMS["n4096"])


def test_handle_lifetime_order(S, ref_or_none):
    sc.handle_lifetime_order(S, *PARAMS["n4096"])


def test_wire_fuzz(S, ref):
    sc.wire_fuzz(S, *PARAMS["n4096"])


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_key_level_order(S, ref, name):
    sc.key_level_order(S, *PARAMS[name])


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_batch_seams(S, ref, name):
    sc.batch_seams(S, *PARAMS[name], count=3)
