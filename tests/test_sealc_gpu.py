"""SEAL-named ABI layer on the real CUDA library (pytest -m gpu): the same FFI sequences as test_sealc_emu.py."""
import ctypes as C
import os

import pytest

import sealc_checks as sc
from params import PARAMS
from sealc_driver import Sealc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def S():
    from sunscreen_b200.lib import B200Lib
    lib = B200Lib.default()
    assert os.path.basename(lib.path) == "libb200bfv.so"
    return Sealc(lib.lib)


def test_simple_multiply_ffi_sequence(S, ref):
    sc.simple_multiply_sequence(S, *PARAMS["n4096"])


@pytest.mark.parametrize("name", ["n4096", "n8192", "n16384"])
def test_evaluator_surface(S, ref_or_none, name):
    sc.evaluator_surface(S, *PARAMS[name])


def test_error_codes(S, ref_or_none):
    sc.error_codes(S, ref_or_none, *PARAMS["n4096"])


def test_batched_multiply_relin_seam(S, ref):
    """B200_Evaluator_MultiplyRelinBatch == per-handle Evaluator_Multiply + Evaluator_Relinearize."""
    import numpy as np
    import refseal
    n, moduli, t = PARAMS["n8192"]
    O = S.context(n, moduli, t)
    inp = refseal.appendix_b_inputs(n, moduli, t)
    rng = np.random.default_rng(2)
    rlk = O.new_ksk({0: inp["rlk"]})
    As, Bs, exp = [], [], []
    for i in range(4):
        a = np.stack([rng.integers(0, moduli[r], size=(2, n), dtype=np.uint64) for r in range(O.k)], axis=1)
        b = np.stack([rng.integers(0, moduli[r], size=(2, n), dtype=np.uint64) for r in range(O.k)], axis=1)
        ha, hb = O.new_ct(a), O.new_ct(b)
        As.append(ha); Bs.append(hb)
        exp.append(O.ct_words(O.relinearize(O.multiply(ha, hb), rlk)))
    dsts = [O._dst() for _ in range(4)]
    vp = C.c_void_p
    O.S.call("B200_Evaluator_MultiplyRelinBatch", O.ev, C.c_uint64(4), (vp * 4)(*As), (vp * 4)(*Bs), rlk, (vp * 4)(*dsts))
    for d, e in zip(dsts, exp):
        assert np.array_equal(O.ct_words(d), e)


def test_bulk_word_access_with_device_buffers(S, ref):
    """B200_Ciphertext_{Set,Get}WordsBatch accept device-resident buffers too (the multi-GPU split hands each rank its
    slice as an NCCL-scattered device tensor, tools/chi_sq_sharded.py): same words as the host-buffer form, and the result
    of MultiplyRelinBatch read back into a device tensor equals the reference's."""
    import numpy as np
    import refseal
    import torch
    n, moduli, t = PARAMS["n8192"]
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    inp = refseal.appendix_b_inputs(n, moduli, t)
    rng = np.random.default_rng(8)
    cnt = 3
    A = np.stack([np.stack([rng.integers(0, moduli[r], size=(2, n), dtype=np.uint64) for r in range(O.k)], axis=1) for _ in range(cnt)])
    B = np.stack([np.stack([rng.integers(0, moduli[r], size=(2, n), dtype=np.uint64) for r in range(O.k)], axis=1) for _ in range(cnt)])
    vp, u64 = C.c_void_p, C.c_uint64
    arr = lambda hs: (vp * len(hs))(*hs)
    dptr = lambda tsr: C.cast(tsr.data_ptr(), C.POINTER(u64))
    dA = torch.from_numpy(A.view(np.int64)).cuda()
    dB = torch.from_numpy(B.view(np.int64)).cuda()
    torch.cuda.synchronize()
    ha, hb, hd = ([O._dst() for _ in range(cnt)] for _ in range(3))
    S.call("B200_Ciphertext_SetWordsBatch", O.ctx, u64(cnt), arr(ha), O.first_id, u64(2), C.c_bool(False), dptr(dA))
    S.call("B200_Ciphertext_SetWordsBatch", O.ctx, u64(cnt), arr(hb), O.first_id, u64(2), C.c_bool(False), dptr(dB))
    for i in range(cnt):
        assert np.array_equal(O.ct_words(ha[i]), A[i]) and np.array_equal(O.ct_words(hb[i]), B[i])
    rlk = O.new_ksk({0: inp["rlk"]})
    S.call("B200_Evaluator_MultiplyRelinBatch", O.ev, u64(cnt), arr(ha), arr(hb), rlk, arr(hd))
    out = torch.zeros((cnt, 2, O.k, n), dtype=torch.int64, device="cuda")
    S.call("B200_Ciphertext_GetWordsBatch", O.ctx, u64(cnt), arr(hd), dptr(out), u64(out.numel()))
    got = out.cpu().numpy().view(np.uint64)
    rrlk = R.new_ksk({0: inp["rlk"]})
    for i in range(cnt):
        exp = R.ct_words(R.relinearize(R.multiply(R.new_ct(A[i]), R.new_ct(B[i])), rrlk))
        assert np.array_equal(got[i], exp), f"item {i}"


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_seeded_encryption_matches_reference(S, ref, name):
    sc.seeded_encryption_parity(S, *PARAMS[name])


@pytest.mark.parametrize("name", ["n4096", "n8192", "n16384"])
def test_keygen_and_encryptor_interoperate_with_reference(S, ref, name):
    sc.keygen_interop(S, *PARAMS[name])


def test_config4_chi_sq_dag_n16384(S, ref):
    """BASELINE config 4 (n=16384, 8 data residues): the chi-squared DAG, word-exact against the reference."""
    sc.chi_sq_dag(S, *PARAMS["n16384"], evaluations=3)


def test_config5_rotate_multiply_plain_sweep_n32768(S, ref_or_none):
    """BASELINE config 5 (n=32768, 15 data residues): rotate_rows + multiply_plain sweep."""
    sc.rotate_multiply_plain_sweep(S, *PARAMS["n32768"], steps=(1, 2, 4, 64, 1024, 8192))


@pytest.mark.parametrize("name", ["n8192", "n16384", "n32768"])
def test_batch_encoder(S, ref_or_none, name):
    sc.batch_encoder_parity(S, *PARAMS[name])


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_wire_format(S, ref, name):
    sc.wire_format(S, *PARAMS[name])


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_polynomial_array(S, ref, name):
    sc.polynomial_array_parity(S, *PARAMS[name])


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_encryption_components(S, ref, name):
    sc.encryption_components_parity(S, *PARAMS[name])


def test_leftover_entry_points(S, ref):
    sc.leftovers_parity(S, *PARAMS["n8192"])


def test_seal_fhe_golden_fixture(S, ref):
    sc.seal_fhe_golden_fixture(S, os.path.join(os.path.dirname(__file__), "golden", "seal_fhe_data"))


@pytest.mark.parametrize("n,moduli,t", [(1024, [0x7e00001], 1 << 8), (2048, [0x3fffffff000001], 65537)])
def test_single_prime_chain(S, ref, n, moduli, t):
    sc.single_prime_context(S, n, moduli, t)


@pytest.mark.parametrize("name", ["n4096", "n8192", "n8192_49", "n16384"])
def test_whole_chain_and_large_sizes(S, ref, name):
    sc.deep_chain_parity(S, *PARAMS[name])


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_misuse_hresults(S, ref, name):
    sc.misuse_hresults(S, *PARAMS[name])


def test_context_validation_sweep(S, ref_or_none):
    sc.context_validation_sweep(S)


def test_concurrent_evaluator_calls(S, ref):
    sc.concurrent_evaluator_calls(S, *PARAMS["n8192"])


def test_combined_calls_isolation(S, ref):
    sc.combined_calls_isolation(S, *PARAMS["n4096"])


def test_handle_lifetime_order(S, ref_or_none):
    sc.handle_lifetime_order(S, *PARAMS["n4096"])


@pytest.mark.parametrize("name", ["n4096", "n8192", "n16384"])
def test_key_level_order(S, ref, name):
    sc.key_level_order(S, *PARAMS[name])


@pytest.mark.parametrize("name", ["n4096", "n8192"])
def test_batch_seams(S, ref, name):
    sc.batch_seams(S, *PARAMS[name], count=9)
