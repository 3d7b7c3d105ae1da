"""CPU-side parity: the product sources compiled in the test-only emulation mode (tests/emu) against the
unmodified reference, on the RNG-free vectors of SURVEY.md App. B.  Covers host precompute, constant folding,
strides and the orchestration of every layer-1 entry point; the CUDA build itself is covered by test_gpu_parity."""
import pytest

import parity_checks as pc
from backends import EmuBackend
from params import PARAMS


@pytest.fixture(scope="module", params=["n4096", "n8192", "n8192_54", "n8192_49"])
def pair(request, emu_lib, ref_or_none):
    n, moduli, t = PARAMS[request.param]
    return pc.Pair(EmuBackend(emu_lib), n, moduli, t)


def test_context_constants(pair):
    pc.check_context(pair)


def test_ntt(pair):
    pc.check_ntt(pair)


def test_elementwise(pair):
    pc.check_elementwise(pair)


def test_multiply_and_relinearize(pair):
    m3 = pc.check_multiply(pair)
    pc.check_relin(pair, m3)


def test_galois(pair):
    if not pair.ctx.using_batching:
        pytest.skip("t does not support batching (reference raises logic_error)")
    pc.check_galois(pair)


def test_plain_ops(pair):
    pc.check_plain(pair)


def test_mod_switch(pair):
    pc.check_modswitch(pair)


def test_adversarial_operands(pair):
    pc.check_adversarial_multiply(pair, with_size5=pair.n <= 4096,
                                  pairs=None if pair.n <= 4096 else [("qm1", "qm1"), ("alt", "pm1"), ("single", "qm1")])
    pc.check_adversarial_keyswitch(pair)


def test_batch_strides(pair):
    if pair.n > 4096:
        pytest.skip("batch stride test runs on the smallest set only (emulation speed)")
    pc.check_batch(pair)


def test_host_buffer_pipeline(pair):
    if pair.n > 4096:
        pytest.skip("host pipeline test runs on the smallest set only (emulation speed)")
    pc.check_host_pipeline(pair)


def test_small_kernels(pair):
    if pair.n > 4096:
        pytest.skip("runs on the smallest set only (emulation speed)")
    pc.check_small_kernels(pair)


def test_noise_norm(pair):
    if pair.n > 4096:
        pytest.skip("noise norm test runs on the smallest set only (emulation speed)")
    pc.check_noise_norm(pair)


def test_encrypted_roundtrip(pair):
    if not pair.ctx.using_batching:
        pytest.skip("needs a batching plain modulus")
    pc.check_encrypted_roundtrip(pair)


def test_n32768_two_level_transform(emu_lib, ref_or_none):
    """BASELINE config 5 parameters (n=32768, 15 data residues + special): the two-level NTT and K=15 kernels."""
    n, moduli, t = PARAMS["n32768"]
    P = pc.Pair(EmuBackend(emu_lib), n, moduli, t)
    pc.check_context(P)
    pc.check_ntt(P, items=1)
    m3 = pc.check_multiply(P, with_sizes=False)
    pc.check_relin(P, m3)
    pc.check_galois(P)
    pc.check_plain(P)
    pc.check_modswitch(P)


def test_layer1_argument_checks(emu_lib):
    """Every layer-1 entry point answers bad arguments (NULL pointers, a level that does not exist, sizes outside the
    supported range, a NULL context) with its error code instead of touching memory."""
    import ctypes as C
    import numpy as np
    from sunscreen_b200.lib import B200Context
    n, moduli, t = PARAMS["n4096"]
    ctx = B200Context(n, moduli, t, lib=emu_lib)
    L, h = emu_lib.lib, ctx.h
    vp, u64, ci = C.c_void_p, C.c_uint64, C.c_int
    k = ctx.k()
    buf = np.zeros((3, k + 1, n), dtype=np.uint64)
    p = vp(buf.ctypes.data)
    E_INVALID, E_NULL = -1, -4
    lv = ctx.first_level
    cases = [
        ("ntt_forward null data", L.b200_ntt_forward, (h, ci(lv), None, u64(1), None), E_NULL),
        ("ntt_forward bad level", L.b200_ntt_forward, (h, ci(99), p, u64(1), None), E_INVALID),
        ("ntt_inverse negative level", L.b200_ntt_inverse, (h, ci(-1), p, u64(1), None), E_INVALID),
        ("ntt_forward null ctx", L.b200_ntt_forward, (None, ci(lv), p, u64(1), None), E_NULL),
        ("add null", L.b200_add, (h, ci(lv), p, None, p, ci(2), u64(1), None), E_NULL),
        ("multiply size 0", L.b200_multiply, (h, ci(lv), p, ci(0), p, ci(2), p, u64(1), None), E_INVALID),
        ("multiply sizes 9 x 9", L.b200_multiply, (h, ci(lv), p, ci(9), p, ci(9), p, u64(1), None), E_INVALID),
        ("multiply null out", L.b200_multiply, (h, ci(lv), p, ci(2), p, ci(2), None, u64(1), None), E_NULL),
        ("square bad level", L.b200_square, (h, ci(7), p, p, u64(1), None), E_INVALID),
        ("relinearize null key", L.b200_relinearize, (h, ci(lv), p, None, p, u64(1), None), E_NULL),
        ("multiply_relin null", L.b200_multiply_relin, (h, ci(lv), p, p, None, p, u64(1), None), E_NULL),
        ("apply_galois even element", L.b200_apply_galois, (h, ci(lv), p, C.c_uint32(4), p, p, u64(1), None), E_INVALID),
        ("apply_galois element too large", L.b200_apply_galois, (h, ci(lv), p, C.c_uint32(2 * n + 1), p, p, u64(1), None), E_INVALID),
        ("multiply_plain null plain", L.b200_multiply_plain, (h, ci(lv), p, ci(2), None, u64(1), p, u64(1), None), E_NULL),
        ("add_plain plain_batch mismatch", L.b200_add_plain, (h, ci(lv), p, ci(2), p, u64(3), p, u64(2), None), E_INVALID),
        ("mod_switch at the last level", L.b200_mod_switch_to_next, (h, ci(ctx.levels - 1), p, ci(2), p, u64(1), None), E_INVALID),
        ("decrypt null", L.b200_decrypt, (h, ci(lv), p, ci(2), None, p, u64(1), None), E_NULL),
        ("decrypt size 1", L.b200_decrypt, (h, ci(lv), p, ci(1), p, p, u64(1), None), E_INVALID),
        ("multiply_relin_host null", L.b200_multiply_relin_host, (h, ci(lv), None, p, p, p, u64(1)), E_NULL),
        ("level_info bad level", L.b200_ctx_level_info, (h, ci(50), p), E_INVALID),
        ("galois_elt_from_step too large", L.b200_galois_elt_from_step, (h, ci(n), p), E_INVALID),
    ]
    wrong = []
    for label, fn, args, want in cases:
        fn.restype = C.c_int
        fn.argtypes = None
        got = fn(*args)
        if got != want:
            wrong.append((label, got, want))
    assert not wrong, wrong
    # zero-sized batches are no-ops
    for fn, args in ((L.b200_ntt_forward, (h, ci(lv), p, u64(0), None)), (L.b200_multiply, (h, ci(lv), p, ci(2), p, ci(2), p, u64(0), None)),
                     (L.b200_multiply_relin, (h, ci(lv), p, p, p, p, u64(0), None))):
        fn.restype = C.c_int
        assert fn(*args) == 0
