"""Pins the plain-C restatement (oracle/bfv_oracle.c) before anything trusts it:
 (a) the reference's own known-answer tests, restated      (tests/seal/util/ntt.cpp:53-133, rns.cpp:460-853)
 (b) the RNG-free golden vectors generated from the unmodified reference (tests/golden/appendix_b.json, small_n64.npz)
 (c) the unmodified reference itself, when oracle/_ref/libsealc_ref.so is present."""
import json
import os

import numpy as np
import pytest

import refseal
from oracle_port import RnsSteps
from params import PARAMS

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "appendix_b.json")))
Q60 = 0xFFFFFFFFFFC0001


# ---- (a) reference KATs --------------------------------------------------------------------------------------
def test_kat_ntt_primitive_roots(port):
    # NTTTablesTest.NTTPrimitiveRootsTest: root_powers[1] at logn=1; [1..3] at logn=2 (bit-reversed powers of psi)
    assert port.min_root(Q60, 2) == 288794978602139552
    psi = port.min_root(Q60, 4)
    # root_powers[bitrev(i)] = psi^i : index 1 = psi^2, index 2 = psi^1, index 3 = psi^3
    assert pow(psi, 2, Q60) == 288794978602139552
    assert psi == 178930308976060547
    assert pow(psi, 3, Q60) == 748001537669050592


def test_kat_negacyclic_ntt(port):
    # NTTTablesTest.NegacyclicNTTTest (n=2)
    assert list(port.ntt_forward(np.array([0, 0], dtype=np.uint64), Q60)) == [0, 0]
    assert list(port.ntt_forward(np.array([1, 0], dtype=np.uint64), Q60)) == [1, 1]
    assert list(port.ntt_forward(np.array([1, 1], dtype=np.uint64), Q60)) == [288794978602139553, 864126526004445282]


def test_kat_inverse_ntt_roundtrip(port):
    # NTTTablesTest.InverseNegacyclicNTTTest (logn=3)
    rng = np.random.default_rng(5)
    assert not port.ntt_inverse(np.zeros(8, dtype=np.uint64), Q60).any()
    for _ in range(20):
        x = rng.integers(0, Q60, size=8, dtype=np.uint64)
        assert np.array_equal(port.ntt_inverse(port.ntt_forward(x, Q60), Q60), x)


def test_kat_fastbconv_m_tilde(port):
    # RNSToolTest.FastBConvMTilde
    r = RnsSteps(port, [3], 2)
    assert r.fastbconv_m_tilde([0, 0]) == [0] * 6
    mt = r.m_tilde
    t1, t2 = mt % 3, (2 * mt) % 3
    base = r.bsk + [mt]
    assert r.fastbconv_m_tilde([1, 2]) == [v % m for m in base for v in (t1, t2)]
    r = RnsSteps(port, [3, 5], 2)
    temp = ((2 * mt) % 3) * 5 + ((4 * mt) % 5) * 3
    base = r.bsk + [mt]
    assert r.fastbconv_m_tilde([1, 1, 2, 2]) == [temp % m for m in base for _ in range(2)]


def test_kat_montgomery_reduction(port):
    # RNSToolTest.MontgomeryReduction
    r = RnsSteps(port, [3], 2)
    mt = r.m_tilde
    assert r.sm_mrq([0] * 6) == [0] * 4
    assert r.sm_mrq([mt, 2 * mt, mt, 2 * mt, 0, 0]) == [1, 2, 1, 2]
    assert r.sm_mrq([3] * 6) == [0] * 4
    r = RnsSteps(port, [3, 5], 2)
    assert r.sm_mrq([mt, 2 * mt] * 3 + [0, 0]) == [1, 2] * 3
    assert r.sm_mrq([15, 30] * 4) == [0] * 6
    assert r.sm_mrq([2 * mt + 15, 2 * mt + 30] * 4) == [2] * 6


def test_kat_fast_floor(port):
    # RNSToolTest.FastFloor
    r = RnsSteps(port, [3], 2)
    assert r.fast_floor([0] * 6) == [0] * 4
    assert r.fast_floor([15, 3] * 3) == [5, 1, 5, 1]
    assert r.fast_floor([17, 4] * 3) == [5, 1, 5, 1]
    r = RnsSteps(port, [3, 5], 2)
    assert r.fast_floor([15, 30] * 5) == [1, 2] * 3
    out = r.fast_floor([21, 32] * 5)
    assert all(abs(e - o) <= 1 for e, o in zip([1, 2] * 3, out))


def test_kat_fastbconv_sk(port):
    # RNSToolTest.FastBConvSK: an integer x given exactly in base Bsk comes back as x mod q
    r = RnsSteps(port, [3], 2)
    assert r.fastbconv_sk([0] * 4) == [0, 0]
    assert r.fastbconv_sk([1, 2, 1, 2]) == [1, 2]
    r = RnsSteps(port, [3, 5], 2)
    assert r.fastbconv_sk([1, 2] * 3) == [1, 2, 1, 2]
    x = [7, 11]
    assert r.fastbconv_sk(x * 3) == [7 % 3, 11 % 3, 7 % 5, 11 % 5]


# ---- (b) golden vectors from the unmodified reference -----------------------------------------------------------
def _port_ops(port, name):
    n, moduli, t = PARAMS[name]
    C = port.context(n, moduli, t)
    inp = refseal.appendix_b_inputs(n, moduli, t)
    return C, inp


@pytest.mark.parametrize("name", ["n4096", "n8192", "n8192_54"])
def test_golden_appendix_b(port, name):
    g = GOLD[name]
    C, inp = _port_ops(port, name)
    n = g["n"]
    H = lambda w: "%016x" % port.fnv(w)
    assert {k: H(v) for k, v in inp.items()} == g["inputs"]
    assert [port.min_root(m, n) for m in g["moduli"]] == g["context"]["roots"]
    aux = C.aux_primes()
    nB = C.base_b_size()
    assert (aux[0], aux[1], nB) == (g["context"]["m_sk"], g["context"]["gamma"], g["context"]["nB"])
    assert aux[2:2 + nB] + [aux[0]] == g["context"]["bsk"]
    ops = g["ops"]
    a, b, p = inp["a"], inp["b"], inp["p"]
    assert H(C.add(a, b)) == ops["add"]
    assert H(C.sub(a, b)) == ops["sub"]
    assert H(C.negate(a)) == ops["negate"]
    m = C.multiply(a, b)
    assert H(m) == ops["multiply"]
    assert H(C.relinearize(m, inp["rlk"])) == ops["relinearize"]
    assert H(C.multiply(a, a)) == ops["square"]
    assert H(C.multiply_plain(a, p)) == ops["multiply_plain"]
    assert H(C.add_plain(a, p)) == ops["add_plain"]
    assert H(C.add_plain(a, p, subtract=True)) == ops["sub_plain"]
    assert H(C.mod_switch_to_next(a)) == ops["mod_switch_to_next"]
    assert H(port.ntt_forward(a[0, 0], g["moduli"][0])) == ops["ntt_a_p0_r0"]
    if ops["rotate_rows_1"]:
        assert C.galois_elt_from_step(1) == 3 and C.galois_elt_from_step(0) == 2 * n - 1
        assert H(C.apply_galois(a, 3, inp["glk3"])) == ops["rotate_rows_1"]
        assert H(C.apply_galois(a, 2 * n - 1, inp["glkc"])) == ops["rotate_columns"]


def test_golden_small_words(port):
    """Word-level fixture at n=64 (three 30-bit primes, t=257): every output word, not just a hash."""
    z = np.load(os.path.join(HERE, "golden", "small_n64.npz"))
    moduli, t = [int(x) for x in z["moduli"]], int(z["t"])
    C = port.context(64, moduli, t)
    a, b, p = z["in_a"], z["in_b"], z["in_p"]
    m = C.multiply(a, b)
    assert np.array_equal(m, z["out_multiply"])
    assert np.array_equal(C.relinearize(m, z["in_rlk"]), z["out_relinearize"])
    assert np.array_equal(C.add(a, b), z["out_add"])
    assert np.array_equal(C.multiply_plain(a, p), z["out_multiply_plain"])
    assert np.array_equal(C.add_plain(a, p), z["out_add_plain"])
    assert np.array_equal(C.apply_galois(a, 3, z["in_glk3"]), z["out_rotate_rows_1"])
    assert np.array_equal(C.apply_galois(a, 127, z["in_glkc"]), z["out_rotate_columns"])
    assert np.array_equal(C.mod_switch_to_next(a), z["out_mod_switch_to_next"])


# ---- (c) against the reference itself ---------------------------------------------------------------------------
def test_against_reference_random(port, ref_or_none):
    """The reference's outputs come from its library when present, else from their records (parity_checks.expect)."""
    from parity_checks import eq, expect
    n, moduli, t = PARAMS["n4096"]
    R = refseal.RefContext(n, moduli, t) if ref_or_none is not None else None
    C = port.context(n, moduli, t)
    rng = np.random.default_rng(9)
    k = len(moduli) - 1
    for trial in range(2):
        a = np.stack([rng.integers(0, moduli[i], size=(2, n), dtype=np.uint64) for i in range(k)], axis=1)
        b = np.stack([rng.integers(0, moduli[i], size=(2, n), dtype=np.uint64) for i in range(k)], axis=1)
        eq(C.multiply(a, b), expect(f"n4096/port multiply, trial {trial}", lambda R: R.ct_words(R.multiply(R.new_ct(a), R.new_ct(b))), R),
           "multiply")
        x = rng.integers(0, moduli[0], size=n, dtype=np.uint64)
        eq(port.ntt_forward(x, moduli[0]), expect(f"n4096/port ntt_forward, trial {trial}", lambda L: L.ntt_forward(moduli[0], x), ref_or_none),
           "ntt_forward")
        eq(port.ntt_inverse(x, moduli[0]), expect(f"n4096/port ntt_inverse, trial {trial}", lambda L: L.ntt_inverse(moduli[0], x), ref_or_none),
           "ntt_inverse")


def test_decrypt_against_reference(port, ref):
    """Fresh keys/encryption from the reference; the port's decrypt (dot product with s + scale&round) returns the
    reference's plaintext."""
    n, moduli, t = PARAMS["n4096"]
    R = refseal.RefContext(n, moduli, t)
    C = port.context(n, moduli, t)
    import ctypes
    kg = R.keygen()
    sk, pk = R.secret_key(kg), R.public_key(kg)
    enc, dec = R.encryptor(pk), R.decryptor(sk)
    msg = np.arange(1, 40, dtype=np.uint64) % t
    ct = R.encrypt(enc, R.new_pt(msg))
    # secret key words: SecretKey_Data -> Plaintext handle (NTT form, key level: K residues)
    h = ctypes.c_void_p()
    R.ref.call("SecretKey_Data", sk, ctypes.byref(h))
    skw = R.pt_coeffs(h).reshape(len(moduli), n)
    got = C.decrypt(R.ct_words(ct), skw[: R.k])
    exp = R.pt_coeffs(R.decrypt(dec, ct))
    assert np.array_equal(got[: exp.size], exp) and not got[exp.size:].any()
