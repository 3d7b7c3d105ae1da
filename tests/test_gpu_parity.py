"""GPU parity (pytest -m gpu): the CUDA library on cuda:0, called through the C ABI, against the unmodified
reference (prebuilt oracle/_ref/libsealc_ref.so) — every output uint64 must be equal."""
import numpy as np
import pytest

import parity_checks as pc
from params import PARAMS

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def be():
    from backends import CudaBackend
    return CudaBackend()


@pytest.fixture(scope="module", params=["n4096", "n8192", "n8192_54", "n8192_49", "n16384", "n32768"])
def pair(request, be, ref_or_none):
    n, moduli, t = PARAMS[request.param]
    return pc.Pair(be, n, moduli, t)


def test_native_library_loaded(be):
    import os
    assert os.path.basename(be.lib.path) == "libb200bfv.so"
    assert be.lib.device_count() >= 1


def test_context_constants(pair):
    pc.check_context(pair)


def test_ntt(pair):
    pc.check_ntt(pair, items=5)


def test_elementwise(pair):
    pc.check_elementwise(pair)


def test_multiply_and_relinearize(pair):
    m3 = pc.check_multiply(pair, with_sizes=pair.n <= 16384)
    pc.check_relin(pair, m3)


def test_galois(pair):
    if not pair.ctx.using_batching:
        pytest.skip("t does not support batching (reference raises logic_error)")
    pc.check_galois(pair)


def test_plain_ops(pair):
    pc.check_plain(pair)


def test_mod_switch(pair):
    pc.check_modswitch(pair)


def test_host_buffer_pipeline(pair):
    if pair.n > 16384:
        pytest.skip("covered at n <= 16384")
    pc.check_host_pipeline(pair, batch=7)


def test_batch_strides(pair):
    pc.check_batch(pair, batch=5 if pair.n <= 16384 else 2)


def test_small_kernels(pair):
    pc.check_small_kernels(pair)


def test_noise_norm(pair):
    pc.check_noise_norm(pair)


def test_encrypted_roundtrip(pair):
    if not pair.ctx.using_batching:
        pytest.skip("needs a batching plain modulus")
    pc.check_encrypted_roundtrip(pair)


def test_adversarial_operands(pair):
    """all-(q-1), alternating, +-1 and single-nonzero operands through multiply / square / multiply_relin / (3,3)->5 and the
    key switch (the 2^53 bound bookkeeping of the FP64 path and its substituted auxiliary base are exercised at their limits)."""
    pc.check_adversarial_multiply(pair, with_size5=pair.n <= 16384,
                                  pairs=None if pair.n <= 16384 else [("qm1", "qm1"), ("alt", "pm1")])
    pc.check_adversarial_keyswitch(pair)


def _threads():
    import os
    return max(1, min(64, len(os.sched_getaffinity(0))))


@pytest.mark.parametrize("name,level", [("n8192", None), ("n8192_54", 0)])
def test_config2_all_16384_transforms_vs_reference(be, ref_or_none, name, level):
    """BASELINE config 2 at FULL size: every one of the 4096 x 4 forward transforms equals the reference's
    ntt_negacyclic_harvey (S/util/ntt.cpp:393-436) word for word (inputs: the fixed-seed splitmix64(0xB200) % q_i generator of
    SURVEY.md App. B); then the inverse returns the input.  Both prime sets of SURVEY.md 8(d): the four default data primes
    (FP64 kernel) and the four 54-bit primes (integer kernel; key level of the {54 x 4} chain)."""
    import refseal
    n, moduli, t = PARAMS[name]
    from sunscreen_b200.lib import B200Context
    ctx = B200Context(n, moduli, t)
    k = ctx.k(level)
    assert k == 4
    items = 4096
    x = np.empty((items, k, n), dtype=np.uint64)
    state = 0xB200
    for i in range(k):
        w, state = refseal.splitmix64_words(items * n, int(moduli[i]), state)
        x[:, i, :] = w.reshape(items, n)
    d = be.to_dev(x)
    ctx.ntt_forward(d, items, level=level)
    got = be.to_host(d)
    R = refseal.RefLib.get() if ref_or_none is not None else None
    for i in range(k):
        label = f"all {items} forward transforms, prime {i}"
        exp = pc.expect(f"{name}/{label}", lambda R: R.ntt_forward_mt(int(moduli[i]), x[:, i, :], _threads()), R)
        pc.eq(got[:, i, :], exp, label)
    ctx.ntt_inverse(d, items, level=level)
    pc.eq(be.to_host(d), x, "inverse of all transforms")


def test_config3_all_1024_pairs_vs_reference(be, ref):
    """BASELINE config 3 at FULL size: 1024 independent pairs of fresh public-key encryptions of batch-encoded uniform
    vectors (reference Encryptor), one relinearization key; multiply + relinearize through b200_multiply_relin (the entry
    point bench.py times) equals the reference's Evaluator::multiply + relinearize_inplace for ALL 1024 pairs, word for word."""
    import refseal
    n, moduli, t = PARAMS["n8192"]
    from sunscreen_b200.lib import B200Context
    ctx = B200Context(n, moduli, t)
    k = ctx.k()
    R = refseal.RefContext(n, moduli, t)
    kg = R.keygen()
    pk, rlk = R.public_key(kg), R.relin_keys(kg)
    enc = R.encryptor(pk)
    benc = R.batch_encoder()
    rng = np.random.default_rng(2024)
    B = 1024
    A = np.empty((B, 2, k, n), dtype=np.uint64)
    Bc = np.empty_like(A)
    for arr in (A, Bc):
        for i in range(B):
            h = R.encrypt(enc, R.batch_encode(benc, rng.integers(0, t, size=n, dtype=np.uint64)))
            arr[i] = R.ct_words(h)
            R.free_ct(h)
    exp = R.mul_relin_batch(A, Bc, rlk, _threads())
    key = R.ksk_words(rlk)[0]
    out = be.empty((B, 2, k, n))
    ctx.multiply_relin(be.to_dev(A), be.to_dev(Bc), be.to_dev(key), out, B)
    got = be.to_host(out)
    for i in range(B):
        if not np.array_equal(got[i], exp[i]):
            pc.eq(got[i], exp[i], f"pair {i} of {B}")


def test_full_size_properties(be):
    """BASELINE config 2/3 sizes through size-independent properties: NTT round trip over 4096x4 polynomials,
    and multiply_relin over a 256-item batch equal to the same items computed one by one."""
    n, moduli, t = PARAMS["n8192"]
    from sunscreen_b200.lib import B200Context
    ctx = B200Context(n, moduli, t)
    k = ctx.k()
    rng = np.random.default_rng(11)
    items = 4096
    x = pc.rand_ct(rng, moduli, k, n, size=1, batch=items)[:, 0]
    d = be.to_dev(x)
    ctx.ntt_forward(d, items)
    f = be.to_host(d)
    assert not np.array_equal(f, x)
    ctx.ntt_inverse(d, items)
    pc.eq(be.to_host(d), x, "4096x4 NTT round trip")
    # linearity of the forward transform: NTT(a+b) = NTT(a)+NTT(b) mod q
    y = pc.rand_ct(rng, moduli, k, n, size=1, batch=8)[:, 0]
    s = np.stack([(x[:8, i].astype(object) + y[:, i].astype(object)) % moduli[i] for i in range(k)], axis=1).astype(np.uint64)
    ds, dy = be.to_dev(s), be.to_dev(y)
    ctx.ntt_forward(ds, 8)
    ctx.ntt_forward(dy, 8)
    fy = be.to_host(dy)
    fs = np.stack([(f[:8, i].astype(object) + fy[:, i].astype(object)) % moduli[i] for i in range(k)], axis=1).astype(np.uint64)
    pc.eq(be.to_host(ds), fs, "NTT linearity")
    B = 256
    A = pc.rand_ct(rng, moduli, k, n, batch=B)
    Bc = pc.rand_ct(rng, moduli, k, n, batch=B)
    key = pc.rand_ksk(rng, moduli, k, n)
    dA, dB, dK = be.to_dev(A), be.to_dev(Bc), be.to_dev(key)
    o = be.empty((B, 2, k, n))
    ctx.multiply_relin(dA, dB, dK, o, B)
    got = be.to_host(o)
    for i in (0, 1, 100, 255):
        oi = be.empty((2, k, n))
        ctx.multiply_relin(be.to_dev(A[i]), be.to_dev(Bc[i]), dK, oi, 1)
        pc.eq(got[i], be.to_host(oi), f"batched item {i} == single")
    # host-buffer entry point returns the same words
    oh = np.zeros((B, 2, k, n), dtype=np.uint64)
    ctx.multiply_relin_host(A, Bc, dK, oh, B)
    pc.eq(oh, got, "multiply_relin_host")
