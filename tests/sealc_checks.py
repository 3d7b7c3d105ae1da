"""Checks of the SEAL-named ABI layer shared by the CPU (emu) and GPU test files."""
import ctypes as C
import json

import numpy as np

import refseal
from parity_checks import eq, expect, param_name
from sealc_driver import Sealc, SealcError

vp, u64 = C.c_void_p, C.c_uint64


def simple_multiply_sequence(S, n, moduli, t, seed=1):
    """examples/simple_multiply through the FFI (SURVEY.md §3.1): keys + fresh encryptions from the reference,
    Evaluator_Multiply (size 3) -> Evaluator_Relinearize (size 2) -> Decryptor_InvariantNoiseBudget -> Decryptor_Decrypt."""
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    assert O.parameters_set
    assert list(O.first_id) == list(R.first_parms_id) and list(O.key_id) == list(R.key_parms_id)
    kg = R.keygen()
    sk, pk, rk = R.secret_key(kg), R.public_key(kg), R.relin_keys(kg)
    enc, dec = R.encryptor(pk), R.decryptor(sk)
    ca, cb = R.encrypt(enc, R.new_pt(np.array([15], dtype=np.uint64))), R.encrypt(enc, R.new_pt(np.array([5], dtype=np.uint64)))
    oa, ob = O.new_ct(R.ct_words(ca)), O.new_ct(R.ct_words(cb))
    ork = O.new_ksk(R.ksk_words(rk))
    rm, om = R.multiply(ca, cb), O.multiply(oa, ob)
    eq(O.ct_words(om), R.ct_words(rm), "Evaluator_Multiply words")
    rr, orr = R.relinearize(rm, rk), O.relinearize(om, ork)
    eq(O.ct_words(orr), R.ct_words(rr), "Evaluator_Relinearize words")
    # decrypt through OUR Decryptor with the reference's secret key words
    h = vp()
    R.ref.call("SecretKey_Data", sk, C.byref(h))
    skw = R.pt_coeffs(h)
    odec = O.decryptor(skw)
    assert O.noise_budget(odec, orr) == R.noise_budget(dec, rr) > 0
    got = O.pt_coeffs(O.decrypt(odec, orr))
    exp = R.pt_coeffs(R.decrypt(dec, rr))
    eq(got, exp, "Decryptor_Decrypt")
    assert int(got[0]) == 75 and got.size == 1


def evaluator_surface(S, n, moduli, t):
    """Every Evaluator entry point seal_fhe uses, on the RNG-free App. B vectors, against the reference's words (the
    reference's values come from its library when present, else from their records: parity_checks.expect)."""
    R = refseal.RefContext(n, moduli, t) if refseal.have_ref() else None
    O = S.context(n, moduli, t)
    inp = refseal.appendix_b_inputs(n, moduli, t)
    oa, ob, op = O.new_ct(inp["a"]), O.new_ct(inp["b"]), O.new_pt(inp["p"])
    orlk = O.new_ksk({0: inp["rlk"]})
    W = lambda h: O.ct_words(h)
    name = param_name(n, moduli, t)

    def ref(label, fn):
        """The reference's ciphertext words of fn(R, a, b, p, rlk) (App. B handles)."""
        return expect(f"{name}/sealc {label}", lambda R: R.ct_words(fn(R, R.new_ct(inp["a"]), R.new_ct(inp["b"]), R.new_pt(inp["p"]),
                                                                        R.new_ksk({0: inp["rlk"]}))), R)
    add_ab = ref("Add", lambda R, a, b, p, k: R.add(a, b))
    eq(W(O.add(oa, ob)), add_ab, "Add")
    eq(W(O.sub(oa, ob)), ref("Sub", lambda R, a, b, p, k: R.sub(a, b)), "Sub")
    eq(W(O.negate(oa)), ref("Negate", lambda R, a, b, p, k: R.negate(a)), "Negate")
    om = O.multiply(oa, ob)
    eq(W(om), ref("Multiply", lambda R, a, b, p, k: R.multiply(a, b)), "Multiply")
    eq(W(O.square(oa)), ref("Square", lambda R, a, b, p, k: R.square(a)), "Square")
    eq(W(O.relinearize(om, orlk)), ref("Relinearize", lambda R, a, b, p, k: R.relinearize(R.multiply(a, b), k)), "Relinearize")
    eq(W(O.add(om, oa)), ref("Add sizes (3,2)", lambda R, a, b, p, k: R.add(R.multiply(a, b), a)), "Add sizes (3,2)")
    eq(W(O.sub(oa, om)), ref("Sub sizes (2,3)", lambda R, a, b, p, k: R.sub(a, R.multiply(a, b))), "Sub sizes (2,3)")
    eq(W(O.multiply_plain(oa, op)), ref("MultiplyPlain", lambda R, a, b, p, k: R.multiply_plain(a, p)), "MultiplyPlain")
    eq(W(O.add_plain(oa, op)), ref("AddPlain", lambda R, a, b, p, k: R.add_plain(a, p)), "AddPlain")
    eq(W(O.sub_plain(oa, op)), ref("SubPlain", lambda R, a, b, p, k: R.sub_plain(a, p)), "SubPlain")
    eq(W(O.mod_switch_to_next(oa)), ref("ModSwitchToNext1", lambda R, a, b, p, k: R.mod_switch_to_next(a)), "ModSwitchToNext1")
    eq(W(O.add_many([oa, ob, oa])), ref("AddMany", lambda R, a, b, p, k: R.add(R.add(a, b), a)), "AddMany")
    # in-place aliasing (evaluator_base.rs:184-196 passes dest == src)
    oc = O.new_ct(inp["a"])
    O.S.call("Evaluator_Add", O.ev, oc, ob, oc)
    eq(W(oc), add_ab, "Add in place")

    # multiply_many / exponentiate: same product tree as the reference (S/evaluator.cpp:1535-1643)
    def multiply_many(R, a, b, p, k):
        d = R.new_ct()
        R.ref.call("Evaluator_MultiplyMany", R.ev, u64(3), (vp * 3)(a, b, a), k, d, None)
        return d

    def exponentiate(R, a, b, p, k):
        d = R.new_ct()
        R.ref.call("Evaluator_Exponentiate", R.ev, a, u64(3), k, d, None)
        return d
    eq(W(O.multiply_many([oa, ob, oa], orlk)), ref("MultiplyMany", multiply_many), "MultiplyMany")
    eq(W(O.exponentiate(oa, 3, orlk)), ref("Exponentiate", exponentiate), "Exponentiate")
    if t % (2 * n) == 1:
        gl = {1: inp["glk3"], (2 * n - 2) // 2: inp["glkc"]}
        og = O.new_ksk(gl)
        eq(W(O.rotate_rows(oa, 1, og)), ref("RotateRows(1)", lambda R, a, b, p, k: R.rotate_rows(a, 1, R.new_ksk(gl))), "RotateRows(1)")
        eq(W(O.rotate_columns(oa, og)), ref("RotateColumns", lambda R, a, b, p, k: R.rotate_columns(a, R.new_ksk(gl))), "RotateColumns")
        # missing key -> NAF decomposition path: steps=3 = 4 - 1 needs keys for +4 and -1; only +1 present -> error like the reference
        for steps in (3,):
            def ref_rotate_code(R):
                try:
                    R.rotate_rows(R.new_ct(inp["a"]), steps, R.new_ksk(gl))
                    return 0
                except refseal.SealError as e:
                    return e.code
            ref_code = expect(f"{name}/sealc RotateRows({steps}) HRESULT", ref_rotate_code, R)
            try:
                O.rotate_rows(oa, steps, og)
                our_code = 0
            except SealcError as e:
                our_code = e.code
            assert our_code == ref_code, (hex(our_code), hex(ref_code))


def error_codes(S, R_lib, n, moduli, t):
    """HRESULT parity with the reference on the failure paths Rust maps (seal_fhe/src/error.rs:65-91); the reference's
    codes come from its library when present (R_lib is not None), else from their records (parity_checks.expect)."""
    O = S.context(n, moduli, t)
    inp = refseal.appendix_b_inputs(n, moduli, t)
    oa = O.new_ct(inp["a"])
    od = O._dst()
    E_POINTER, E_INVALIDARG, E_INVOP = 0x80004003, 0x80070057, 0x80131509

    def ref_codes(R_lib):
        R = refseal.RefContext(n, moduli, t)
        ra, rd, re = R.new_ct(inp["a"]), R.new_ct(), R.new_ct()
        rk_empty = vp()
        R.ref.call("KSwitchKeys_Create1", C.byref(rk_empty))
        codes = {"NULL destination": R.ref.call_rc("Evaluator_Multiply", R.ev, ra, ra, None, None),
                 "empty operand": R.ref.call_rc("Evaluator_Multiply", R.ev, re, ra, rd, None),
                 "transparent result": R.ref.call_rc("Evaluator_Sub", R.ev, ra, ra, rd),
                 "missing keys": R.ref.call_rc("Evaluator_Relinearize", R.ev, R.multiply(ra, ra), rk_empty, rd, None)}
        R.ref.call("Ciphertext_SetIsNTTForm", ra, C.c_bool(True))
        codes["NTT-form input"] = R.ref.call_rc("Evaluator_Multiply", R.ev, ra, ra, rd, None)
        return codes
    ref = expect(f"{param_name(n, moduli, t)}/sealc error codes", ref_codes, R_lib)
    # NULL handle
    assert O.S.rc("Evaluator_Multiply", O.ev, oa, oa, None, None) == ref["NULL destination"] == E_POINTER
    assert O.S.rc("Evaluator_Add", None, oa, oa, od) == E_POINTER
    # empty operand
    oe = O._dst()
    assert O.S.rc("Evaluator_Multiply", O.ev, oe, oa, od, None) == ref["empty operand"] == E_INVALIDARG
    # transparent result: a - a
    assert O.S.rc("Evaluator_Sub", O.ev, oa, oa, od) == ref["transparent result"] == E_INVOP
    # relinearize with keys of the wrong parms_id / missing keys
    ok_empty = vp()
    O.S.call("KSwitchKeys_Create1", C.byref(ok_empty))
    om = O.multiply(oa, oa)
    assert O.S.rc("Evaluator_Relinearize", O.ev, om, ok_empty, od, None) == ref["missing keys"] == E_INVALIDARG
    # NTT-form input to multiply
    O.S.call("Ciphertext_SetIsNTTForm", oa, C.c_bool(True))
    assert O.S.rc("Evaluator_Multiply", O.ev, oa, oa, od, None) == ref["NTT-form input"] == E_INVALIDARG
    # invalid parameters: context reports parameters not set, Evaluator_Create fails
    bad = S.context(n, [moduli[0], moduli[0] + 2], t, sec=0)
    assert not bad.parameters_set
    ev = vp()
    assert S.rc("Evaluator_Create", bad.ctx, C.byref(ev)) == E_INVALIDARG


def _ref_pk_words(R, pk):
    h = vp()
    R.ref.call("PublicKey_Data", pk, C.byref(h))
    return R.ct_words_any(h)


def seeded_encryption_parity(S, n, moduli, t):
    """pk-encryption from a fixed 64-byte seed: our B200_Encryptor_EncryptSetSeed reproduces the reference's
    Encryptor_EncryptReturnComponentsSetSeed ciphertext word for word (same Blake2xb stream, same samplers)."""
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    kg = R.keygen()
    pk = R.public_key(kg)
    pkw = _ref_pk_words(R, pk)
    enc_r = R.encryptor(pk)
    # our Encryptor over the same public key words
    opk = vp()
    O.S.call("PublicKey_Create1", C.byref(opk))
    opk_ct = vp()
    O.S.call("PublicKey_Data", opk, C.byref(opk_ct))
    w = np.ascontiguousarray(pkw, dtype=np.uint64)
    O.S.call("B200_Ciphertext_SetWords", opk_ct, O.ctx, O.key_id, u64(2), C.c_bool(True), w.ctypes.data_as(C.POINTER(u64)))
    enc_o = vp()
    O.S.call("Encryptor_Create", O.ctx, opk, None, C.byref(enc_o))
    rng = np.random.default_rng(4)
    for trial, seed in enumerate(([0] * 8, [1, 2, 3, 4, 5, 6, 7, 8], list(rng.integers(0, 2**63, size=8)))):
        msg = rng.integers(0, t, size=n if trial else 3, dtype=np.uint64)
        seed_arr = (u64 * 8)(*[int(x) for x in seed])
        # reference
        rct = R.new_ct()
        pa_u, pa_e, rem = vp(), vp(), vp()
        R.ref.call("PolynomialArray_Create", None, C.byref(pa_u))
        R.ref.call("PolynomialArray_Create", None, C.byref(pa_e))
        R.ref.call("Plaintext_Create1", None, C.byref(rem))
        R.ref.call("Encryptor_EncryptReturnComponentsSetSeed", enc_r, R.new_pt(msg), C.c_bool(False), rct, pa_u, pa_e, rem,
                   seed_arr, None)
        # ours
        oct_ = O._dst()
        O.S.call("B200_Encryptor_EncryptSetSeed", enc_o, O.new_pt(msg), seed_arr, oct_)
        eq(O.ct_words(oct_), R.ct_words(rct), f"seeded encryption, trial {trial}")


def keygen_interop(S, n, moduli, t):
    """Keys made by OUR KeyGenerator (host sampling + GPU arithmetic) are valid keys for the REFERENCE: a ciphertext
    encrypted by our Encryptor is multiplied / relinearized / rotated by the reference's Evaluator with our keys and
    decrypted by the reference's Decryptor with our secret key — and the same through our own layer."""
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    kg = vp()
    O.S.call("KeyGenerator_Create1", O.ctx, C.byref(kg))
    sk, pk, rlk = vp(), vp(), vp()
    O.S.call("KeyGenerator_SecretKey", kg, C.byref(sk))
    O.S.call("KeyGenerator_CreatePublicKey", kg, C.c_bool(False), C.byref(pk))
    O.S.call("KeyGenerator_CreateRelinKeys", kg, C.c_bool(False), C.byref(rlk))
    # secret key words -> reference SecretKey
    skd = vp()
    O.S.call("SecretKey_Data", sk, C.byref(skd))
    skw = O.pt_coeffs(skd)
    rsk = vp()
    R.ref.call("SecretKey_Create1", C.byref(rsk))
    rskd = vp()
    R.ref.call("SecretKey_Data", rsk, C.byref(rskd))
    R.ref.call("Plaintext_Resize", rskd, u64(skw.size))
    C.memmove(R.ref.lib.refshim_pt_data(rskd), skw.ctypes.data, skw.nbytes)
    R.ref.call("Plaintext_SetParmsId", rskd, R.key_parms_id)
    rdec = R.decryptor(rsk)
    # relin keys -> reference
    cnt = u64()
    O.S.call("KSwitchKeys_GetKeyList", rlk, u64(0), C.byref(cnt), None)
    lst = (vp * cnt.value)()
    O.S.call("KSwitchKeys_GetKeyList", rlk, u64(0), C.byref(cnt), lst)
    words = []
    for h in lst:
        d = vp()
        O.S.call("PublicKey_Data", vp(h), C.byref(d))
        words.append(O.ct_words_key(d))
    rrlk = R.new_ksk({0: np.stack(words)})
    # encrypt with OUR encryptor (pk) and symmetric encryptor (sk)
    enc = vp()
    O.S.call("Encryptor_Create", O.ctx, pk, sk, C.byref(enc))
    rng = np.random.default_rng(8)
    m1 = rng.integers(0, t, size=n, dtype=np.uint64)
    m2 = rng.integers(0, t, size=16, dtype=np.uint64)
    c1, c2 = O._dst(), O._dst()
    O.S.call("Encryptor_Encrypt", enc, O.new_pt(m1), c1, None)
    O.S.call("Encryptor_EncryptSymmetric", enc, O.new_pt(m2), C.c_bool(False), c2, None)
    r1, r2 = R.new_ct(O.ct_words(c1)), R.new_ct(O.ct_words(c2))
    assert R.noise_budget(rdec, r1) > 20 and R.noise_budget(rdec, r2) > 20
    eq(R.pt_coeffs(R.decrypt(rdec, r1)), m1[: np.flatnonzero(m1)[-1] + 1], "reference decrypts our pk-encryption")
    eq(R.pt_coeffs(R.decrypt(rdec, r2)), m2[: np.flatnonzero(m2)[-1] + 1], "reference decrypts our sk-encryption")
    # reference evaluator with OUR relin keys: (c1 * c2) relinearized decrypts to the negacyclic product mod t
    rprod = R.relinearize(R.multiply(r1, r2), rrlk)
    assert R.noise_budget(rdec, rprod) > 0
    exp = np.zeros(n, dtype=object)
    for i, a in enumerate(m2):
        if a:
            shifted = np.concatenate([-(m1[n - i:].astype(object)), m1[: n - i].astype(object)]) if i else m1.astype(object)
            exp = (exp + int(a) * shifted) % t
    got = R.pt_coeffs(R.decrypt(rdec, rprod)).astype(object)
    full = np.zeros(n, dtype=object)
    full[: got.size] = got
    assert np.array_equal(full, exp % t), "product under our relinearization keys decrypts wrongly on the reference"
    # and entirely inside our layer
    odec = O.decryptor(skw)
    oprod = O.relinearize(O.multiply(c1, c2), rlk)
    eq(O.ct_words(oprod), R.ct_words(rprod), "our evaluator == reference evaluator on our keys")
    got2 = np.zeros(n, dtype=object)
    g = O.pt_coeffs(O.decrypt(odec, oprod)).astype(object)
    got2[: g.size] = g
    assert np.array_equal(got2, exp % t)
    if t % (2 * n) == 1:
        glk = vp()
        steps = (C.c_int * 2)(1, -2)
        O.S.call("KeyGenerator_CreateGaloisKeysFromSteps", kg, u64(2), steps, C.c_bool(False), C.byref(glk))
        be_ = R.batch_encoder()
        vals = rng.integers(0, t, size=n, dtype=np.uint64)
        cv = O._dst()
        O.S.call("Encryptor_Encrypt", enc, O.new_pt(R.pt_coeffs(R.batch_encode(be_, vals))), cv, None)
        rot = O.rotate_rows(cv, 1, glk)
        back = R.batch_decode(be_, R.decrypt(rdec, R.new_ct(O.ct_words(rot))))
        half = n // 2
        expect = np.concatenate([np.roll(vals[:half], -1), np.roll(vals[half:], -1)])
        eq(back, expect, "rotate_rows(1) with our Galois keys")


def chi_sq_dag(S, n, moduli, t, evaluations=2):
    """BASELINE config 4: the optimised chi-squared circuit (examples/chi_sq/src/main.rs:59-88) as the DAG
    sunscreen_runtime executes it — every Multiply followed by the Relinearize the compiler inserts
    (sunscreen_backend/src/transforms/insert_relinearizations.rs:17-62) — replayed through both C ABIs on the same
    fresh encryptions; every output ciphertext word must match, and the outputs decrypt to the plain computation."""
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    kg = R.keygen()
    sk, pk, rk = R.secret_key(kg), R.public_key(kg), R.relin_keys(kg)
    enc, dec = R.encryptor(pk), R.decryptor(sk)
    ork = O.new_ksk(R.ksk_words(rk))
    rng = np.random.default_rng(12)

    def circuit(E, rlk, n0, n1, n2):
        mul = lambda a, b: E.relinearize(E.multiply(a, b), rlk)
        x = E.add(E.add(n0, n0), n1)
        y = E.add(E.add(n2, n2), n1)
        a = mul(n0, n2)
        a = E.add(a, a)
        a = E.add(a, a)
        alpha = E.sub(a, mul(n1, n1))
        alpha = mul(alpha, alpha)
        b1 = mul(x, x)
        b1 = E.add(b1, b1)
        b2 = mul(x, y)
        b3 = mul(y, y)
        b3 = E.add(b3, b3)
        return alpha, b1, b2, b3

    for _ in range(evaluations):
        vals = [int(v) for v in rng.integers(1, 12, size=3)]
        rin = [R.encrypt(enc, R.new_pt(np.array([v], dtype=np.uint64))) for v in vals]
        oin = [O.new_ct(R.ct_words(h)) for h in rin]
        rout = circuit(R, rk, *rin)
        oout = circuit(O, ork, *oin)
        n0, n1, n2 = vals
        x, y = 2 * n0 + n1, 2 * n2 + n1
        expect = [(4 * n0 * n2 - n1 * n1) ** 2, 2 * x * x, x * y, 2 * y * y]
        for name, hr, ho, e in zip(("alpha", "b_1", "b_2", "b_3"), rout, oout, expect):
            eq(O.ct_words(ho), R.ct_words(hr), f"chi_sq output {name}")
            got = R.pt_coeffs(R.decrypt(dec, R.new_ct(O.ct_words(ho))))
            assert int(got[0]) == e % t and got.size == 1, (name, got[:4], e)


def rotate_multiply_plain_sweep(S, n, moduli, t, steps=(1, 2, 4, 64)):
    """BASELINE config 5: rotate_rows by powers of two followed by multiply_plain with a dense plaintext, with
    Galois keys for exactly those steps, against the reference word for word (the reference's words come from its library
    when present, else from their records: parity_checks.expect)."""
    R = refseal.RefContext(n, moduli, t) if refseal.have_ref() else None
    O = S.context(n, moduli, t)
    inp = refseal.appendix_b_inputs(n, moduli, t)
    name = param_name(n, moduli, t)
    rng = np.random.default_rng(21)
    K = len(moduli)
    k = K - 1 if K > 1 else 1
    keys = {}
    for s in steps:
        elt = pow(3, s, 2 * n)
        key = np.empty((k, 2, K, n), dtype=np.uint64)
        for i in range(K):
            key[:, :, i, :] = rng.integers(0, moduli[i], size=(k, 2, n), dtype=np.uint64)
        keys[(elt - 1) // 2] = key
    og = O.new_ksk(keys)
    oa, op = O.new_ct(inp["a"]), O.new_pt(inp["p"])

    def ref_rotate(s, then_plain):
        def fn(R):
            rr = R.rotate_rows(R.new_ct(inp["a"]), s, R.new_ksk(keys))
            return R.ct_words(R.multiply_plain(rr, R.new_pt(inp["p"])) if then_plain else rr)
        return fn
    for s in steps:
        orr = O.rotate_rows(oa, s, og)
        eq(O.ct_words(orr), expect(f"{name}/sealc rotate_rows({s})", ref_rotate(s, False), R), f"rotate_rows({s})")
        label = f"multiply_plain after rotate_rows({s})"
        eq(O.ct_words(O.multiply_plain(orr, op)), expect(f"{name}/sealc {label}", ref_rotate(s, True), R), label)


def batch_encoder_parity(S, n, moduli, t):
    """BatchEncoder_Encode/Decode (slot permutation + negacyclic NTT mod t) against the reference (its values come from
    its library when present, else from their records: parity_checks.expect)."""
    R = refseal.RefContext(n, moduli, t) if refseal.have_ref() else None
    O = S.context(n, moduli, t)
    name = param_name(n, moduli, t)
    obe = vp()
    O.S.call("BatchEncoder_Create", O.ctx, C.byref(obe))
    cnt = u64()
    O.S.call("BatchEncoder_GetSlotCount", obe, C.byref(cnt))
    assert cnt.value == n
    rng = np.random.default_rng(33)
    for size in (n, 7, 0):
        vals = rng.integers(0, t, size=size, dtype=np.uint64)
        op = vp()
        O.S.call("Plaintext_Create1", None, C.byref(op))
        O.S.call("BatchEncoder_Encode1", obe, u64(size), vals.ctypes.data_as(C.POINTER(u64)), op)
        label = f"BatchEncoder_Encode1 ({size} values)"
        eq(O.pt_coeffs(op), expect(f"{name}/sealc {label}", lambda R: R.pt_coeffs(R.batch_encode(R.batch_encoder(), vals)), R), label)
        out = np.zeros(n, dtype=np.uint64)
        c2 = u64(n)
        O.S.call("BatchEncoder_Decode1", obe, op, C.byref(c2), out.ctypes.data_as(C.POINTER(u64)), None)
        exp = np.zeros(n, dtype=np.uint64)
        exp[:size] = vals
        eq(out, exp, "BatchEncoder_Decode1 round trip")
    # signed variant
    sv = rng.integers(-(t // 2), t // 2, size=n, dtype=np.int64)
    op = vp()
    O.S.call("Plaintext_Create1", None, C.byref(op))
    O.S.call("BatchEncoder_Encode2", obe, u64(n), sv.ctypes.data_as(C.POINTER(C.c_int64)), op)

    def ref_encode2(R):
        rp = vp()
        R.ref.call("Plaintext_Create1", None, C.byref(rp))
        R.ref.call("BatchEncoder_Encode2", R.batch_encoder(), u64(n), sv.ctypes.data_as(C.POINTER(C.c_int64)), rp)
        return R.pt_coeffs(rp)
    eq(O.pt_coeffs(op), expect(f"{name}/sealc BatchEncoder_Encode2", ref_encode2, R), "BatchEncoder_Encode2")
    so = np.zeros(n, dtype=np.int64)
    c2 = u64(n)
    O.S.call("BatchEncoder_Decode2", obe, op, C.byref(c2), so.ctypes.data_as(C.POINTER(C.c_int64)), None)
    assert np.array_equal(so, sv)


# ------------------------------------------------------------------------------------------------------------
# wire format, PolynomialArray, component-returning encryption, small leftovers of the seal_fhe surface
# ------------------------------------------------------------------------------------------------------------
COMPR_NONE, COMPR_ZLIB, COMPR_ZSTD = 0, 1, 2
E_INVALIDARG, COR_E_INVALIDOPERATION, COR_E_IO, E_POINTER = 0x80070057, 0x80131509, 0x80131620, 0x80004003
_CREATE = {"Ciphertext": ("Ciphertext_Create1", True), "Plaintext": ("Plaintext_Create1", True),
           "PublicKey": ("PublicKey_Create1", False), "SecretKey": ("SecretKey_Create1", False),
           "KSwitchKeys": ("KSwitchKeys_Create1", False)}


class _Lib:
    """Uniform view of `call` / `rc` over the reference (RefLib) and our Sealc driver."""

    def __init__(self, call, rc, ctx):
        self.call, self.rc, self.ctx = call, rc, ctx

    def new(self, kind):
        name, pool = _CREATE[kind]
        h = vp()
        self.call(name, None, C.byref(h)) if pool else self.call(name, C.byref(h))
        return h

    def save_size(self, kind, h, mode):
        r = C.c_int64()
        self.call(kind + "_SaveSize", h, C.c_uint8(mode), C.byref(r))
        return r.value

    def save(self, kind, h, mode):
        cap = self.save_size(kind, h, mode)
        buf = (C.c_uint8 * cap)()
        n = C.c_int64()
        self.call(kind + "_Save", h, buf, u64(cap), C.c_uint8(mode), C.byref(n))
        assert 16 <= n.value <= cap
        return bytes(buf[: n.value])

    def load_rc(self, kind, h, data, unsafe=False):
        n = C.c_int64()
        buf = (C.c_uint8 * max(len(data), 1)).from_buffer_copy(data if data else b"\0")
        rc = self.rc(kind + ("_UnsafeLoad" if unsafe else "_Load"), h, self.ctx, buf, u64(len(data)), C.byref(n))
        return rc, n.value

    def load(self, kind, data, unsafe=False):
        h = self.new(kind)
        rc, n = self.load_rc(kind, h, data, unsafe)
        assert rc == 0, f"{kind}_Load -> 0x{rc:08x}"
        assert n == len(data)
        return h


def _libs(R, O):
    return _Lib(R.ref.call, R.ref.call_rc, R.ctx), _Lib(O.S.call, O.S.rc, O.ctx)


def wire_format(S, n, moduli, t):
    """Save / SaveSize / Load of every data object: byte-identical to the reference with compr_mode none, and
    interchangeable with it in both directions with zlib and Zstandard; the same HRESULTs on malformed input."""
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    RL, OL = _libs(R, O)
    kg = R.keygen()
    sk, pk, rlk = R.secret_key(kg), R.public_key(kg), R.relin_keys(kg)
    glk = R.galois_keys_steps(kg, [1]) if t % (2 * n) == 1 else None
    enc = R.encryptor(pk, sk)
    rng = np.random.default_rng(11)
    msg = rng.integers(0, t, size=n // 2 + 3, dtype=np.uint64)
    pt = R.new_pt(msg)
    ct = R.encrypt(enc, pt)
    ct3 = R.multiply(ct, ct)
    empty_ct = R.new_ct()
    objs = [("Ciphertext", ct), ("Ciphertext", ct3), ("Plaintext", pt), ("Plaintext", R.new_pt(np.zeros(0, dtype=np.uint64))), ("PublicKey", pk),
            ("SecretKey", sk), ("KSwitchKeys", rlk)]
    if glk is not None:
        objs.append(("KSwitchKeys", glk))
    for kind, h in objs:
        raw = RL.save(kind, h, COMPR_NONE)
        assert RL.save_size(kind, h, COMPR_NONE) == len(raw)
        ours = OL.load(kind, raw)
        assert OL.save_size(kind, ours, COMPR_NONE) == len(raw)
        assert OL.save(kind, ours, COMPR_NONE) == raw, f"{kind}: Save(none) differs from the reference"
        for mode in (COMPR_ZLIB, COMPR_ZSTD):
            assert OL.save_size(kind, ours, mode) == RL.save_size(kind, h, mode)
            # reference -> ours
            z_ref = RL.save(kind, h, mode)
            assert OL.save(kind, OL.load(kind, z_ref), COMPR_NONE) == raw, f"{kind}: cannot read the reference's mode {mode}"
            # ours -> reference
            z_our = OL.save(kind, ours, mode)
            assert len(z_our) < len(raw) or len(raw) < 256
            assert RL.save(kind, RL.load(kind, z_our), COMPR_NONE) == raw, f"{kind}: reference cannot read our mode {mode}"
    # seeded symmetric ciphertext (S/util/rlwe.cpp:441-457 -> S/ciphertext.cpp:118-151,204-224): half-size on the wire,
    # expanded from the stored PRNG seed when loaded
    sct = R.new_ct()
    R.ref.call("Encryptor_EncryptSymmetric", enc, pt, C.c_bool(True), sct, None)
    sraw = RL.save("Ciphertext", sct, COMPR_NONE)
    full = RL.save("Ciphertext", ct, COMPR_NONE)
    assert len(sraw) < 0.6 * len(full)
    ref_expanded = RL.save("Ciphertext", RL.load("Ciphertext", sraw), COMPR_NONE)
    assert len(ref_expanded) == len(full)
    assert OL.save("Ciphertext", OL.load("Ciphertext", sraw), COMPR_NONE) == ref_expanded, "seed expansion differs"
    # ---- HRESULTs on bad input, side by side ----
    raw_ct = RL.save("Ciphertext", ct, COMPR_NONE)
    raw_pk = RL.save("PublicKey", pk, COMPR_NONE)
    bad_magic = b"\x00\x00" + raw_ct[2:]
    bad_version = raw_ct[:3] + b"\x09" + raw_ct[4:]
    bad_mode = raw_ct[:5] + b"\x07" + raw_ct[6:]
    big = bytearray(raw_ct)
    off = len(raw_ct) - 8  # last coefficient of the last residue polynomial
    big[off:off + 8] = (2**63).to_bytes(8, "little")
    wrong_size = bytearray(raw_ct)
    wrong_size[16 + 33:16 + 41] = (9).to_bytes(8, "little")  # the size_ member
    raw_empty = RL.save("Ciphertext", empty_ct, COMPR_NONE)
    assert OL.save("Ciphertext", OL.new("Ciphertext"), COMPR_NONE) == raw_empty, "empty ciphertext serialises differently"
    cases = [("empty ciphertext", "Ciphertext", raw_empty, False), ("empty ciphertext, unsafe", "Ciphertext", raw_empty, True),
             ("truncated", "Ciphertext", raw_ct[:-5], False), ("too short", "Ciphertext", raw_ct[:10], False),
             ("bad magic", "Ciphertext", bad_magic, False), ("bad version", "Ciphertext", bad_version, False),
             ("bad compr mode", "Ciphertext", bad_mode, False), ("coefficient out of range", "Ciphertext", bytes(big), False),
             ("coefficient out of range, unsafe", "Ciphertext", bytes(big), True), ("size member 9", "Ciphertext", bytes(wrong_size), False),
             ("key-level ct via Ciphertext_Load", "Ciphertext", raw_pk, False),
             ("key-level ct via Ciphertext_UnsafeLoad", "Ciphertext", raw_pk, True),
             ("ct bytes via Plaintext_Load", "Plaintext", raw_ct, False), ("ct bytes via KSwitchKeys_Load", "KSwitchKeys", raw_ct, False),
             ("zstd garbage", "Ciphertext", raw_ct[:5] + b"\x02" + raw_ct[6:], False),
             ("zlib garbage", "Ciphertext", raw_ct[:5] + b"\x01" + raw_ct[6:], False)]
    for label, kind, data, unsafe in cases:
        r_rc, _ = RL.load_rc(kind, RL.new(kind), data, unsafe)
        o_rc, _ = OL.load_rc(kind, OL.new(kind), data, unsafe)
        assert o_rc == r_rc, f"{label}: ours 0x{o_rc:08x}, reference 0x{r_rc:08x}"
    for L in (RL, OL):
        r = C.c_int64()
        assert L.rc("Ciphertext_SaveSize", L.load("Ciphertext", raw_ct), C.c_uint8(9), C.byref(r)) == E_INVALIDARG
        buf = (C.c_uint8 * len(raw_ct))()
        h = L.load("Ciphertext", raw_ct)
        assert L.rc("Ciphertext_Save", h, buf, u64(len(raw_ct)), C.c_uint8(9), C.byref(r)) == E_INVALIDARG
        assert L.rc("Ciphertext_Save", h, buf, u64(8), C.c_uint8(0), C.byref(r)) == E_INVALIDARG
        assert L.rc("Ciphertext_Save", h, buf, u64(len(raw_ct) - 1), C.c_uint8(0), C.byref(r)) == COR_E_IO


def _pa_export(L, h):
    vals = {}
    for name in ("ExportSize", "PolySize", "PolyModulusDegree", "CoeffModulusSize"):
        v = u64()
        L.call("PolynomialArray_" + name, h, C.byref(v))
        vals[name] = v.value
    for name in ("IsReserved", "IsRns", "IsMultiprecision"):
        b = C.c_bool()
        L.call("PolynomialArray_" + name, h, C.byref(b))
        vals[name] = b.value
    out = np.zeros(vals["ExportSize"], dtype=np.uint64)
    if out.size:
        L.call("PolynomialArray_PerformExport", h, out.ctypes.data_as(C.POINTER(u64)))
    return vals, out


def _pa_same(RL, OL, rh, oh, what):
    rv, rw = _pa_export(RL, rh)
    ov, ow = _pa_export(OL, oh)
    assert ov == rv, f"{what}: {ov} vs {rv}"
    eq(ow, rw, what)


def polynomial_array_parity(S, n, moduli, t):
    """PolynomialArray_* (the fork's container for proof inputs): construction from ciphertext / public key / secret key,
    RNS <-> multi-precision conversion, Drop and Copy give the reference's words."""
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    RL, OL = _libs(R, O)
    kg = R.keygen()
    sk, pk = R.secret_key(kg), R.public_key(kg)
    ct = R.encrypt(R.encryptor(pk), R.new_pt(np.arange(1, 40, dtype=np.uint64) % t))
    blobs = {"Ciphertext": RL.save("Ciphertext", ct, 0), "PublicKey": RL.save("PublicKey", pk, 0), "SecretKey": RL.save("SecretKey", sk, 0)}
    for kind, raw in blobs.items():
        oh_src = OL.load(kind, raw)
        rh_src = {"Ciphertext": ct, "PublicKey": pk, "SecretKey": sk}[kind]
        rh, oh = vp(), vp()
        RL.call("PolynomialArray_CreateFrom" + kind, None, R.ctx, rh_src, C.byref(rh))
        OL.call("PolynomialArray_CreateFrom" + kind, None, O.ctx, oh_src, C.byref(oh))
        _pa_same(RL, OL, rh, oh, f"PolynomialArray from {kind}")
        rc_, oc_ = vp(), vp()
        RL.call("PolynomialArray_Copy", rh, C.byref(rc_))
        OL.call("PolynomialArray_Copy", oh, C.byref(oc_))
        _pa_same(RL, OL, rc_, oc_, f"Copy of {kind} array")
        if kind != "SecretKey":
            rd, od = vp(), vp()
            RL.call("PolynomialArray_Drop", rh, C.byref(rd))
            OL.call("PolynomialArray_Drop", oh, C.byref(od))
            _pa_same(RL, OL, rd, od, f"Drop of {kind} array")
        RL.call("PolynomialArray_ToMultiprecision", rh)
        OL.call("PolynomialArray_ToMultiprecision", oh)
        _pa_same(RL, OL, rh, oh, f"{kind} array in multi-precision form")
        RL.call("PolynomialArray_ToRns", rh)
        OL.call("PolynomialArray_ToRns", oh)
        _pa_same(RL, OL, rh, oh, f"{kind} array back in RNS form")
        RL.call("PolynomialArray_Destroy", rh)
        OL.call("PolynomialArray_Destroy", oh)
    # an unreserved array
    rh, oh = vp(), vp()
    RL.call("PolynomialArray_Create", None, C.byref(rh))
    OL.call("PolynomialArray_Create", None, C.byref(oh))
    _pa_same(RL, OL, rh, oh, "fresh PolynomialArray")


def encryption_components_parity(S, n, moduli, t):
    """Encryptor_Encrypt{,Symmetric}ReturnComponentsSetSeed: ciphertext, u, e and the rounding remainder all equal the
    reference's for the same seed, with and without the special modulus."""
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    RL, OL = _libs(R, O)
    kg = R.keygen()
    sk, pk = R.secret_key(kg), R.public_key(kg)
    renc = R.encryptor(pk, sk)
    opk, osk = OL.load("PublicKey", RL.save("PublicKey", pk, 0)), OL.load("SecretKey", RL.save("SecretKey", sk, 0))
    oenc = vp()
    O.S.call("Encryptor_Create", O.ctx, opk, osk, C.byref(oenc))
    rng = np.random.default_rng(21)
    for trial in range(3):
        msg = rng.integers(0, t, size=(5, n, n // 3)[trial], dtype=np.uint64)
        seed = (u64 * 8)(*[int(x) for x in rng.integers(0, 2**63, size=8)])
        for disable in (False, True):
            outs = []
            for L, encryptor, new_pt in ((RL, renc, R.new_pt), (OL, oenc, O.new_pt)):
                ct, u, e, rem = L.new("Ciphertext"), vp(), vp(), L.new("Plaintext")
                L.call("PolynomialArray_Create", None, C.byref(u))
                L.call("PolynomialArray_Create", None, C.byref(e))
                L.call("Encryptor_EncryptReturnComponentsSetSeed", encryptor, new_pt(msg), C.c_bool(disable), ct, u, e, rem, seed, None)
                outs.append((L.save("Ciphertext", ct, 0), _pa_export(L, u), _pa_export(L, e), L.save("Plaintext", rem, 0)))
            (rct, ru, re_, rrem), (oct_, ou, oe, orem) = outs
            assert oct_ == rct, f"asymmetric ciphertext differs (disable_special_modulus={disable})"
            assert ou[0] == ru[0] and oe[0] == re_[0]
            eq(ou[1], ru[1], "u component")
            eq(oe[1], re_[1], "e component")
            assert orem == rrem, "remainder differs"
        # Symmetric variant.  The reference does NOT forward the seed on this path (S/encryptor.cpp:225-236 calls
        # encrypt_zero_symmetric without it, S/util/rlwe.h:128-143), so its output is random even with SetSeed; ours
        # honours the seed.  Checked: the reference really is non-deterministic here, ours is deterministic, the
        # remainder matches, the exported noise is a clipped Gaussian sample with consistent residues, and the
        # reference decrypts our ciphertext.
        def sym(L, encryptor, new_pt):
            ct, e, rem = L.new("Ciphertext"), vp(), L.new("Plaintext")
            L.call("PolynomialArray_Create", None, C.byref(e))
            L.call("Encryptor_EncryptSymmetricReturnComponentsSetSeed", encryptor, new_pt(msg), ct, e, rem, seed, None)
            return L.save("Ciphertext", ct, 0), _pa_export(L, e), L.save("Plaintext", rem, 0)
        r1, r2 = sym(RL, renc, R.new_pt), sym(RL, renc, R.new_pt)
        o1, o2 = sym(OL, oenc, O.new_pt), sym(OL, oenc, O.new_pt)
        assert r1[0] != r2[0], "the reference's symmetric SetSeed path became deterministic: compare words instead"
        assert o1[0] == o2[0] and np.array_equal(o1[1][1], o2[1][1])
        assert o1[2] == r1[2], "remainder differs"
        assert o1[1][0] == r1[1][0], "shape of the exported noise differs"
        k = R.k
        ev = o1[1][1].reshape(k, n)
        signed = [np.where(ev[i] > moduli[i] // 2, ev[i].astype(np.int64) - np.int64(moduli[i]), ev[i].astype(np.int64)) for i in range(k)]
        assert all(np.array_equal(signed[0], s) for s in signed) and np.abs(signed[0]).max() <= 19 and np.abs(signed[0]).max() >= 3
        back = R.pt_coeffs(R.decrypt(R.decryptor(sk), RL.load("Ciphertext", o1[0])))
        eq(back, msg[: np.flatnonzero(msg)[-1] + 1], "reference decrypts our seeded symmetric encryption")
    # unseeded variants run and decrypt
    dec = R.decryptor(sk)
    for name, args in (("Encryptor_EncryptReturnComponents", lambda ct, u, e, rem: (C.c_bool(False), ct, u, e, rem, None)),
                       ("Encryptor_EncryptSymmetricReturnComponents", lambda ct, u, e, rem: (ct, e, rem, None))):
        ct, u, e, rem = OL.new("Ciphertext"), vp(), vp(), OL.new("Plaintext")
        OL.call("PolynomialArray_Create", None, C.byref(u))
        OL.call("PolynomialArray_Create", None, C.byref(e))
        msg = rng.integers(1, t, size=17, dtype=np.uint64)
        OL.call(name, oenc, O.new_pt(msg), *args(ct, u, e, rem))
        back = R.pt_coeffs(R.decrypt(dec, RL.load("Ciphertext", OL.save("Ciphertext", ct, 0))))
        eq(back, msg, name)


def leftovers_parity(S, n, moduli, t):
    """Plaintext_Create4 (hex polynomial strings), Evaluator_ModSwitchToNext2 (NTT-form plaintexts) and
    Decryptor_InvariantNoise (double), each against the reference: values and HRESULTs."""
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    RL, OL = _libs(R, O)
    for s in ("", "0", "1", "7FFx^3 + 1x^1 + 3", "1x^4095", "ABCDEFabcdef0123x^2", "1x^2 + 2x^2", "1x^1 + 2x^2", "3 + 1x^1", "x^2",
              "1x^", "1 x^2", "1x^2+3", "00000000000000000001x^1", "10000000000000000x^1", "FFFFFFFFFFFFFFFFx^1 + 0", "1x^3 + ",
              "Gx^1", "2x^1 + 0x^0"):
        rh, oh = vp(), vp()
        r_rc = RL.rc("Plaintext_Create4", s.encode(), None, C.byref(rh))
        o_rc = OL.rc("Plaintext_Create4", s.encode(), None, C.byref(oh))
        assert o_rc == r_rc, f"Plaintext_Create4({s!r}): ours 0x{o_rc:08x}, reference 0x{r_rc:08x}"
        if r_rc == 0:
            eq(O.pt_coeffs(oh), R.pt_coeffs(rh), f"Plaintext_Create4({s!r})")
    # an NTT-form plaintext at the first data level: k*n residues + parms_id
    k = R.k
    rng = np.random.default_rng(2)
    words = np.concatenate([rng.integers(0, moduli[i], size=n, dtype=np.uint64) for i in range(k)])
    outs = []
    for L, first_id, make in ((RL, R.first_parms_id, R.new_pt), (OL, O.first_id, O.new_pt)):
        p = make(words)
        L.call("Plaintext_SetParmsId", p, first_id)
        d = L.new("Plaintext")
        ev = R.ev if L is RL else O.ev
        rc = L.rc("Evaluator_ModSwitchToNext2", ev, p, d)
        plain = make(np.array([1, 2, 3], dtype=np.uint64))
        rc_plain = L.rc("Evaluator_ModSwitchToNext2", ev, plain, L.new("Plaintext"))
        bad = make(words + np.uint64(2**62))
        L.call("Plaintext_SetParmsId", bad, first_id)
        rc_bad = L.rc("Evaluator_ModSwitchToNext2", ev, bad, L.new("Plaintext"))
        outs.append((rc, rc_plain, rc_bad, L.save("Plaintext", d, 0) if rc == 0 else None))
    assert outs[0] == outs[1], f"ModSwitchToNext2: reference {outs[0][:3]}, ours {outs[1][:3]}"
    # invariant noise as a double
    kg = R.keygen()
    sk, pk, rlk = R.secret_key(kg), R.public_key(kg), R.relin_keys(kg)
    ct = R.encrypt(R.encryptor(pk), R.new_pt(np.array([3, 1, 4, 1, 5], dtype=np.uint64)))
    prod = R.relinearize(R.multiply(ct, ct), rlk)
    osk = OL.load("SecretKey", RL.save("SecretKey", sk, 0))
    rdec, odec = R.decryptor(sk), vp()
    O.S.call("Decryptor_Create", O.ctx, osk, C.byref(odec))
    for h in (ct, prod):
        oh = OL.load("Ciphertext", RL.save("Ciphertext", h, 0))
        a, b = C.c_double(), C.c_double()
        RL.call("Decryptor_InvariantNoise", rdec, h, C.byref(a))
        OL.call("Decryptor_InvariantNoise", odec, oh, C.byref(b))
        assert a.value == b.value and 0.0 < a.value < 0.5, (a.value, b.value)


def _siphash13(data):
    """Rust's DefaultHasher (SipHash-1-3, zero keys) over `data`."""
    M = (1 << 64) - 1
    rotl = lambda x, b: ((x << b) | (x >> (64 - b))) & M
    v = [0x736f6d6570736575, 0x646f72616e646f6d, 0x6c7967656e657261, 0x7465646279746573]

    def rnd():
        v[0] = (v[0] + v[1]) & M; v[1] = rotl(v[1], 13) ^ v[0]; v[0] = rotl(v[0], 32)
        v[2] = (v[2] + v[3]) & M; v[3] = rotl(v[3], 16) ^ v[2]
        v[0] = (v[0] + v[3]) & M; v[3] = rotl(v[3], 21) ^ v[0]
        v[2] = (v[2] + v[1]) & M; v[1] = rotl(v[1], 17) ^ v[2]; v[2] = rotl(v[2], 32)

    nbytes = len(data)
    for m in np.frombuffer(data[: nbytes - nbytes % 8], dtype="<u8").tolist():
        v[3] ^= m; rnd(); v[0] ^= m
    b = (nbytes & 0xff) << 56
    for i, ch in enumerate(data[nbytes - nbytes % 8:]):
        b |= ch << (8 * i)
    v[3] ^= b; rnd(); v[0] ^= b
    v[2] ^= 0xff; rnd(); rnd(); rnd()
    return v[0] ^ v[1] ^ v[2] ^ v[3]


def seal_fhe_golden_fixture(S, golden_dir):
    """seal_fhe's own deterministic-encryption test (seal_fhe/src/encryptor_decryptor.rs:886-932) replayed through the FFI:
    the fixture keys (tests/data/{public,secret}_key.bin, Zstandard) load, encrypt_deterministic(seed 0) of 0..8191 gives
    the reference's ciphertext word for word — and the reference's serialisation of it hashes to the crate's golden value."""
    import os
    n, bits = 8192, [50, 30, 30, 50, 50]
    Rl = refseal.RefLib.get()
    ctxs = []
    for call in (Rl.call, S.call):
        arr = (vp * len(bits))()
        call("CoeffModulus_Create1", u64(n), u64(len(bits)), (C.c_int * len(bits))(*bits), arr)
        mods = []
        for h in arr:
            v = u64()
            call("Modulus_Value", vp(h), C.byref(v))
            mods.append(v.value)
        pm = (vp * 1)()
        call("CoeffModulus_Create1", u64(n), u64(1), (C.c_int * 1)(20), pm)
        tv = u64()
        call("Modulus_Value", vp(pm[0]), C.byref(tv))
        parms, ctx = vp(), vp()
        call("EncParams_Create1", C.c_uint8(1), C.byref(parms))
        call("EncParams_SetPolyModulusDegree", parms, u64(n))
        call("EncParams_SetCoeffModulus", parms, u64(len(bits)), arr)
        call("EncParams_SetPlainModulus2", parms, tv)
        call("SEALContext_Create", parms, C.c_bool(False), C.c_int(128), C.byref(ctx))
        ctxs.append((mods, tv.value, ctx))
    assert ctxs[0][:2] == ctxs[1][:2], "CoeffModulus_Create1 / PlainModulus::batching primes differ"
    assert ctxs[0][1] == 1032193
    RL, OL = _Lib(Rl.call, Rl.call_rc, ctxs[0][2]), _Lib(S.call, S.rc, ctxs[1][2])
    pkb = open(os.path.join(golden_dir, "public_key.bin"), "rb").read()
    skb = open(os.path.join(golden_dir, "secret_key.bin"), "rb").read()
    results = []
    for L in (RL, OL):
        last = (u64 * 4)()
        first = (u64 * 4)()
        L.call("SEALContext_LastParmsId", L.ctx, last)
        L.call("SEALContext_FirstParmsId", L.ctx, first)
        assert list(last) == list(first), "expand_mod_chain = false: the chain ends at the first data level"
        pk, sk = L.load("PublicKey", pkb), L.load("SecretKey", skb)
        be, enc, dec = vp(), vp(), vp()
        L.call("BatchEncoder_Create", L.ctx, C.byref(be))
        L.call("Encryptor_Create", L.ctx, pk, sk, C.byref(enc))
        L.call("Decryptor_Create", L.ctx, sk, C.byref(dec))
        vals = (u64 * n)(*range(n))
        pt = L.new("Plaintext")
        L.call("BatchEncoder_Encode1", be, u64(n), vals, pt)
        ct, u, e, rem = L.new("Ciphertext"), vp(), vp(), L.new("Plaintext")
        L.call("PolynomialArray_Create", None, C.byref(u))
        L.call("PolynomialArray_Create", None, C.byref(e))
        L.call("Encryptor_EncryptReturnComponentsSetSeed", enc, pt, C.c_bool(False), ct, u, e, rem, (u64 * 8)(), None)
        out = L.new("Plaintext")
        L.call("Decryptor_Decrypt", dec, ct, out)
        cnt = u64(n)
        back = (u64 * n)()
        L.call("BatchEncoder_Decode1", be, out, C.byref(cnt), back, None)
        assert list(back) == list(range(n))
        results.append((L.save("PublicKey", pk, 0), L.save("SecretKey", sk, 0), L.save("Ciphertext", ct, 0), ct))
    assert results[0][0] == results[1][0] and results[0][1] == results[1][1], "fixture keys decode differently"
    assert results[0][2] == results[1][2], "deterministic encryption differs from the reference"
    # the crate's golden value pins the REFERENCE build (its vendored zstd 1.4.5 included); our Zstandard bytes come from
    # the system library, so for our side the check is that the reference reads them back to the same ciphertext
    zref = RL.save("Ciphertext", results[0][3], COMPR_ZSTD)
    assert _siphash13(len(zref).to_bytes(8, "little") + zref) == 9942548233613012008
    zour = OL.save("Ciphertext", results[1][3], COMPR_ZSTD)
    assert RL.save("Ciphertext", RL.load("Ciphertext", zour), 0) == results[0][2]
    # a build that compiled the Zstandard 1.4.5 the reference vendors into the library (csrc/Makefile: B200_VENDORED_ZSTD)
    # emits the reference's bytes exactly: the crate's own `deterministic` test would then see its golden hash
    has = getattr(S.lib, "B200_VendoredZstd", None)
    if has is not None and has() == 1:
        assert zour == zref, "vendored Zstandard 1.4.5: compressed ciphertext bytes differ from the reference's"
        assert _siphash13(len(zour).to_bytes(8, "little") + zour) == 9942548233613012008
        for kind, idx in (("PublicKey", 0), ("SecretKey", 1)):
            ro, oo = (L.load(kind, results[i][idx]) for i, L in ((0, RL), (1, OL)))
            assert RL.save(kind, ro, COMPR_ZSTD) == OL.save(kind, oo, COMPR_ZSTD), f"{kind}: Zstandard bytes differ"


def single_prime_context(S, n, moduli, t):
    """Chains of ONE prime (BFVDefault for n = 1024 / 2048): no key level above the data level, no key switching
    (S/context.cpp:478-497: using_keyswitching() is false).  Encryption, addition, ciphertext x ciphertext multiplication
    (size 3, cannot be relinearized), plain operations and decryption of the size-3 result agree with the reference; asking
    for relinearization keys fails the same way."""
    assert len(moduli) == 1
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    assert O.parameters_set
    assert list(O.first_id) == list(R.first_parms_id) == list(O.key_id) == list(R.key_parms_id)
    RL, OL = _libs(R, O)
    for L in (RL, OL):
        b = C.c_bool(True)
        L.call("SEALContext_UsingKeyswitching", L.ctx, C.byref(b))
        assert b.value is False
    kg = R.keygen()
    sk, pk = R.secret_key(kg), R.public_key(kg)
    okg, orl = vp(), vp()
    O.S.call("KeyGenerator_Create1", O.ctx, C.byref(okg))
    rrl = vp()
    r_rc = RL.rc("KeyGenerator_CreateRelinKeys", kg, C.c_bool(False), C.byref(rrl))
    o_rc = OL.rc("KeyGenerator_CreateRelinKeys", okg, C.c_bool(False), C.byref(orl))
    assert r_rc == o_rc != 0, (hex(r_rc), hex(o_rc))
    enc, dec = R.encryptor(pk, sk), R.decryptor(sk)
    rng = np.random.default_rng(5)
    m1 = rng.integers(0, t, size=n, dtype=np.uint64)
    m2 = rng.integers(0, min(t, 4), size=5, dtype=np.uint64)
    m2[-1] = 1
    c1, c2 = R.encrypt(enc, R.new_pt(m1)), R.encrypt(enc, R.new_pt(m2))
    o1, o2 = OL.load("Ciphertext", RL.save("Ciphertext", c1, 0)), OL.load("Ciphertext", RL.save("Ciphertext", c2, 0))

    def same(rh, oh, what):
        eq(np.frombuffer(OL.save("Ciphertext", oh, 0), dtype=np.uint8), np.frombuffer(RL.save("Ciphertext", rh, 0), dtype=np.uint8), what)

    same(R.add(c1, c2), O.add(o1, o2), "add (single prime)")
    same(R.sub(c1, c2), O.sub(o1, o2), "sub (single prime)")
    rm, om = R.multiply(c1, c2), O.multiply(o1, o2)
    same(rm, om, "multiply (single prime, size 3)")
    same(R.square(c2), O.square(o2), "square (single prime)")
    pt = rng.integers(1, t, size=7, dtype=np.uint64)
    same(R.multiply_plain(c1, R.new_pt(pt)), O.multiply_plain(o1, O.new_pt(pt)), "multiply_plain (single prime)")
    same(R.add_plain(c1, R.new_pt(pt)), O.add_plain(o1, O.new_pt(pt)), "add_plain (single prime)")
    # decrypt the size-3 product with OUR decryptor and the reference's
    osk = OL.load("SecretKey", RL.save("SecretKey", sk, 0))
    odec = vp()
    O.S.call("Decryptor_Create", O.ctx, osk, C.byref(odec))
    out = OL.new("Plaintext")
    O.S.call("Decryptor_Decrypt", odec, om, out)
    eq(O.pt_coeffs(out), R.pt_coeffs(R.decrypt(dec, rm)), "decrypt size-3 (single prime)")
    nb_r, nb_o = C.c_int(), C.c_int()
    RL.call("Decryptor_InvariantNoiseBudget", dec, rm, C.byref(nb_r))
    OL.call("Decryptor_InvariantNoiseBudget", odec, om, C.byref(nb_o))
    assert nb_r.value == nb_o.value
    # our own keys / encryptions on such a context decrypt on the reference
    opk, oenc, osk2 = vp(), vp(), vp()
    O.S.call("KeyGenerator_SecretKey", okg, C.byref(osk2))
    O.S.call("KeyGenerator_CreatePublicKey", okg, C.c_bool(False), C.byref(opk))
    O.S.call("Encryptor_Create", O.ctx, opk, osk2, C.byref(oenc))
    oc = OL.new("Ciphertext")
    O.S.call("Encryptor_Encrypt", oenc, O.new_pt(m2), oc, None)
    rsk = RL.load("SecretKey", OL.save("SecretKey", osk2, 0))
    rdec2 = R.decryptor(rsk)
    eq(R.pt_coeffs(R.decrypt(rdec2, RL.load("Ciphertext", OL.save("Ciphertext", oc, 0)))), m2, "reference decrypts our encryption (single prime)")


def deep_chain_parity(S, n, moduli, t):
    """The rest of the modulus-switching chain and the larger ciphertext sizes: at EVERY data level (down to one
    residue) multiply / square / relinearize / rotate / plain operations / decrypt agree word for word with the reference;
    products of size-3 operands (sizes 4 and 5), their sums, and the HRESULTs of what cannot be done with them
    (relinearize without s^3 keys, rotate a size-3 ciphertext, switch below the last level)."""
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    RL, OL = _libs(R, O)
    kg = R.keygen()
    sk, pk, rlk = R.secret_key(kg), R.public_key(kg), R.relin_keys(kg)
    batching = t % (2 * n) == 1
    glk = R.galois_keys_steps(kg, [1, 4, -1]) if batching else None
    enc, dec = R.encryptor(pk, sk), R.decryptor(sk)
    orlk = OL.load("KSwitchKeys", RL.save("KSwitchKeys", rlk, 0))
    oglk = OL.load("KSwitchKeys", RL.save("KSwitchKeys", glk, 0)) if batching else None
    osk = OL.load("SecretKey", RL.save("SecretKey", sk, 0))
    odec = vp()
    O.S.call("Decryptor_Create", O.ctx, osk, C.byref(odec))
    rng = np.random.default_rng(31)
    to_ours = lambda h: OL.load("Ciphertext", RL.save("Ciphertext", h, 0))

    def same(rh, oh, what):
        a, b = OL.save("Ciphertext", oh, 0), RL.save("Ciphertext", rh, 0)
        assert a == b, f"{what}: serialised ciphertexts differ"

    def rc_pair(name, r_args, o_args):
        r, o = RL.rc(name, *r_args), OL.rc(name, *o_args)
        assert r == o, f"{name}: reference 0x{r:08x}, ours 0x{o:08x}"
        return r

    ra = R.encrypt(enc, R.new_pt(rng.integers(0, t, size=n, dtype=np.uint64)))
    rb = R.encrypt(enc, R.new_pt(rng.integers(0, t, size=n // 2, dtype=np.uint64)))
    oa, ob = to_ours(ra), to_ours(rb)
    pl = rng.integers(1, t, size=n, dtype=np.uint64)
    level = 0
    while True:
        tag = f"level +{level}"
        rm, om = R.multiply(ra, rb), O.multiply(oa, ob)
        same(rm, om, f"multiply, {tag}")
        same(R.square(ra), O.square(oa), f"square, {tag}")
        rr, orr = R.relinearize(rm, rlk), O.relinearize(om, orlk)
        same(rr, orr, f"relinearize, {tag}")
        same(R.multiply_plain(ra, R.new_pt(pl)), O.multiply_plain(oa, O.new_pt(pl)), f"multiply_plain, {tag}")
        same(R.add_plain(rb, R.new_pt(pl)), O.add_plain(ob, O.new_pt(pl)), f"add_plain, {tag}")
        same(R.sub_plain(rb, R.new_pt(pl)), O.sub_plain(ob, O.new_pt(pl)), f"sub_plain, {tag}")
        if batching:
            same(R.rotate_rows(ra, 1, glk), O.rotate_rows(oa, 1, oglk), f"rotate_rows(1), {tag}")
            same(R.rotate_rows(ra, 3, glk), O.rotate_rows(oa, 3, oglk), f"rotate_rows(3) via its NAF 4 - 1, {tag}")
        out = OL.new("Plaintext")
        O.S.call("Decryptor_Decrypt", odec, orr, out)
        eq(O.pt_coeffs(out), R.pt_coeffs(R.decrypt(dec, rr)), f"decrypt, {tag}")
        assert O.noise_budget(odec, orr) == R.noise_budget(dec, rr)
        if level == 0:
            # sizes 4 and 5
            r4, o4 = R.multiply(rm, rb), O.multiply(om, ob)
            same(r4, o4, "multiply (3,2) -> 4")
            r5, o5 = R.multiply(rm, rm), O.multiply(om, om)
            same(r5, o5, "multiply (3,3) -> 5")
            same(R.square(rm), O.square(om), "square of a size-3 ciphertext (falls back to multiply)")
            same(R.add(r5, r4), O.add(o5, o4), "add (5,4)")
            same(R.sub(r4, r5), O.sub(o4, o5), "sub (4,5)")
            same(R.negate(r5), O.negate(o5), "negate size 5")
            out = OL.new("Plaintext")
            O.S.call("Decryptor_Decrypt", odec, o4, out)
            eq(O.pt_coeffs(out), R.pt_coeffs(R.decrypt(dec, r4)), "decrypt size 4")
            assert rc_pair("Evaluator_Relinearize", (R.ev, r4, rlk, RL.new("Ciphertext"), None), (O.ev, o4, orlk, OL.new("Ciphertext"), None)) != 0
            if batching:
                assert rc_pair("Evaluator_RotateRows", (R.ev, rm, C.c_int(1), glk, RL.new("Ciphertext"), None),
                               (O.ev, om, C.c_int(1), oglk, OL.new("Ciphertext"), None)) != 0
            # the reference multiplies anything up to a destination of SEAL_CIPHERTEXT_SIZE_MAX = 16 polynomials (the noise
            # budget is long gone; the words are still a deterministic function of the inputs)
            r9, o9 = R.multiply(r5, r5), O.multiply(o5, o5)
            same(r9, o9, "multiply (5,5) -> 9")
            assert rc_pair("Evaluator_Multiply", (R.ev, r9, r9, RL.new("Ciphertext"), None), (O.ev, o9, o9, OL.new("Ciphertext"), None)) != 0
        # next level (operands of different levels must be rejected alike)
        rn, on = RL.new("Ciphertext"), OL.new("Ciphertext")
        rc = rc_pair("Evaluator_ModSwitchToNext1", (R.ev, ra, rn, None), (O.ev, oa, on, None))
        if rc != 0:
            break
        same(rn, on, f"mod_switch_to_next, {tag}")
        assert rc_pair("Evaluator_Add", (R.ev, ra, rn, RL.new("Ciphertext")), (O.ev, oa, on, OL.new("Ciphertext"))) != 0
        rbn, obn = RL.new("Ciphertext"), OL.new("Ciphertext")
        rc_pair("Evaluator_ModSwitchToNext1", (R.ev, rb, rbn, None), (O.ev, ob, obn, None))
        ra, oa, rb, ob = rn, on, rbn, obn
        level += 1
    assert level == len(moduli) - 2, "the chain should end at a single residue"


def key_level_order(S, n, moduli, t):
    """One RelinKeys / GaloisKeys object used FIRST at the lowest level that still key-switches and THEN at the first level
    (and through the batch seam): the cached device copy of a key must serve every level in any order (a cache sized
    by the first use returned garbage for the later, higher-level use)."""
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    RL, OL = _libs(R, O)
    kg = R.keygen()
    sk, pk, rlk = R.secret_key(kg), R.public_key(kg), R.relin_keys(kg)
    batching = t % (2 * n) == 1
    glk = R.galois_keys_steps(kg, [1]) if batching else None
    enc = R.encryptor(pk)
    orlk = OL.load("KSwitchKeys", RL.save("KSwitchKeys", rlk, 0))
    oglk = OL.load("KSwitchKeys", RL.save("KSwitchKeys", glk, 0)) if batching else None
    rng = np.random.default_rng(77)
    ra = R.encrypt(enc, R.new_pt(rng.integers(0, t, size=n, dtype=np.uint64)))
    rb = R.encrypt(enc, R.new_pt(rng.integers(0, t, size=n, dtype=np.uint64)))
    oa, ob = (OL.load("Ciphertext", RL.save("Ciphertext", h, 0)) for h in (ra, rb))
    same = lambda rh, oh, what: eq(np.frombuffer(OL.save("Ciphertext", oh, 0), dtype=np.uint8),
                                   np.frombuffer(RL.save("Ciphertext", rh, 0), dtype=np.uint8), what)
    # walk both operands down to the last level
    chain = [(ra, rb, oa, ob)]
    for _ in range(len(moduli) - 2):
        ra_, rb_, oa_, ob_ = chain[-1]
        chain.append((R.mod_switch_to_next(ra_), R.mod_switch_to_next(rb_), O.mod_switch_to_next(oa_), O.mod_switch_to_next(ob_)))
    for idx in list(range(len(chain) - 1, -1, -1)) + [len(chain) - 1, 0]:
        ra_, rb_, oa_, ob_ = chain[idx]
        same(R.relinearize(R.multiply(ra_, rb_), rlk), O.relinearize(O.multiply(oa_, ob_), orlk), f"relinearize, level +{idx}")
        if batching:
            same(R.rotate_rows(ra_, 1, glk), O.rotate_rows(oa_, 1, oglk), f"rotate_rows, level +{idx}")
        d = OL.new("Ciphertext")
        O.S.call("B200_Evaluator_MultiplyRelinBatch", O.ev, u64(1), (vp * 1)(oa_), (vp * 1)(ob_), orlk, (vp * 1)(d))
        same(R.relinearize(R.multiply(ra_, rb_), rlk), d, f"MultiplyRelinBatch, level +{idx}")


def misuse_hresults(S, n, moduli, t):
    """A sweep of calls the Rust wrappers can make with bad arguments: both libraries must answer every one of them with
    the same HRESULT (and leave the same values where there are any)."""
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    RL, OL = _libs(R, O)
    kg = R.keygen()
    sk, pk, rlk = R.secret_key(kg), R.public_key(kg), R.relin_keys(kg)
    enc = R.encryptor(pk, sk)
    msg = np.arange(1, 9, dtype=np.uint64)
    rct = R.encrypt(enc, R.new_pt(msg))
    blob = {"ct": RL.save("Ciphertext", rct, 0), "pk": RL.save("PublicKey", pk, 0), "sk": RL.save("SecretKey", sk, 0),
            "rlk": RL.save("KSwitchKeys", rlk, 0)}
    mismatches = []

    def both(label, fn):
        """fn(L, objs) -> (hresult or tuple); compared across the two libraries"""
        res = []
        for L, ev in ((RL, R.ev), (OL, O.ev)):
            objs = {"ct": L.load("Ciphertext", blob["ct"]), "pk": L.load("PublicKey", blob["pk"]), "sk": L.load("SecretKey", blob["sk"]),
                    "rlk": L.load("KSwitchKeys", blob["rlk"]), "ev": ev, "dst": L.new("Ciphertext"), "pt": L.new("Plaintext")}
            try:
                res.append(fn(L, objs))
            except Exception as e:  # a helper raised: record its text so that both sides must raise alike
                res.append(("raised", type(e).__name__, str(e)[-40:]))
        if res[0] != res[1]:
            mismatches.append(f"{label}: reference {res[0]}, ours {res[1]}")

    def new_pt(L, coeffs):
        h = L.new("Plaintext")
        L.call("Plaintext_Resize", h, u64(len(coeffs)))
        for i, v in enumerate(coeffs):
            L.call("Plaintext_SetCoeffAt", h, u64(i), u64(int(v)))
        return h

    # plaintext operands that are not valid for the parameters
    both("AddPlain, coefficient >= t", lambda L, o: L.rc("Evaluator_AddPlain", o["ev"], o["ct"], new_pt(L, [t]), o["dst"]))
    both("MultiplyPlain, coefficient >= t", lambda L, o: L.rc("Evaluator_MultiplyPlain", o["ev"], o["ct"], new_pt(L, [1, t + 5]), o["dst"], None))
    both("MultiplyPlain by zero", lambda L, o: L.rc("Evaluator_MultiplyPlain", o["ev"], o["ct"], new_pt(L, [0, 0]), o["dst"], None))
    both("MultiplyPlain by empty plaintext", lambda L, o: L.rc("Evaluator_MultiplyPlain", o["ev"], o["ct"], o["pt"], o["dst"], None))
    both("AddPlain with empty plaintext", lambda L, o: (L.rc("Evaluator_AddPlain", o["ev"], o["ct"], o["pt"], o["dst"]), L.save("Ciphertext", o["dst"], 0)))
    both("SubPlain, too many coefficients", lambda L, o: L.rc("Evaluator_SubPlain", o["ev"], o["ct"], new_pt(L, [1] * (n + 1)), o["dst"]))
    # plaintext accessors
    both("Plaintext_CoeffAt out of range", lambda L, o: L.rc("Plaintext_CoeffAt", new_pt(L, [1, 2]), u64(5), C.byref(u64())))
    both("Plaintext_SetCoeffAt out of range", lambda L, o: L.rc("Plaintext_SetCoeffAt", new_pt(L, [1, 2]), u64(2), u64(1)))
    both("Plaintext_Resize beyond n then encrypt", lambda L, o: L.rc("Evaluator_AddPlain", o["ev"], o["ct"], new_pt(L, [0] * (2 * n)), o["dst"]))
    # ciphertext accessors
    both("Ciphertext_GetDataAt1 out of range", lambda L, o: L.rc("Ciphertext_GetDataAt1", o["ct"], u64(10**9), C.byref(u64())))
    both("Ciphertext_GetDataAt2 poly out of range", lambda L, o: L.rc("Ciphertext_GetDataAt2", o["ct"], u64(2), u64(0), C.byref(u64())))
    both("Ciphertext_GetDataAt2 coeff out of range", lambda L, o: L.rc("Ciphertext_GetDataAt2", o["ct"], u64(1), u64(10**9), C.byref(u64())))
    both("Ciphertext accessors on an empty ciphertext", lambda L, o: tuple(
        (L.rc(name, o["dst"], C.byref(v)), v.value) for name, v in (("Ciphertext_Size", u64(7)), ("Ciphertext_CoeffModulusSize", u64(7)), ("Ciphertext_PolyModulusDegree", u64(7)))))
    # evaluator on empty / mismatched operands
    both("Negate of an empty ciphertext", lambda L, o: L.rc("Evaluator_Negate", o["ev"], o["dst"], L.new("Ciphertext")))
    both("Square of an empty ciphertext", lambda L, o: L.rc("Evaluator_Square", o["ev"], o["dst"], L.new("Ciphertext"), None))
    both("Relinearize of a size-2 ciphertext", lambda L, o: (L.rc("Evaluator_Relinearize", o["ev"], o["ct"], o["rlk"], o["dst"], None), L.save("Ciphertext", o["dst"], 0)))
    both("Relinearize with an empty key object", lambda L, o: L.rc("Evaluator_Relinearize", o["ev"], o["ct"], L.new("KSwitchKeys"), o["dst"], None))
    both("RotateRows with relinearization keys", lambda L, o: L.rc("Evaluator_RotateRows", o["ev"], o["ct"], C.c_int(1), o["rlk"], o["dst"], None))
    both("RotateRows by 0", lambda L, o: (L.rc("Evaluator_RotateRows", o["ev"], o["ct"], C.c_int(0), o["rlk"], o["dst"], None),))
    both("RotateRows by n", lambda L, o: L.rc("Evaluator_RotateRows", o["ev"], o["ct"], C.c_int(n), o["rlk"], o["dst"], None))
    both("Exponentiate to the power 0", lambda L, o: L.rc("Evaluator_Exponentiate", o["ev"], o["ct"], u64(0), o["rlk"], o["dst"], None))
    both("Exponentiate to the power 1", lambda L, o: (L.rc("Evaluator_Exponentiate", o["ev"], o["ct"], u64(1), o["rlk"], o["dst"], None), L.save("Ciphertext", o["dst"], 0)))
    both("MultiplyMany of nothing", lambda L, o: L.rc("Evaluator_MultiplyMany", o["ev"], u64(0), (vp * 1)(), o["rlk"], o["dst"], None))
    both("AddMany of nothing", lambda L, o: L.rc("Evaluator_AddMany", o["ev"], u64(0), (vp * 1)(), o["dst"]))
    both("AddMany of one", lambda L, o: (L.rc("Evaluator_AddMany", o["ev"], u64(1), (vp * 1)(o["ct"]), o["dst"]), L.save("Ciphertext", o["dst"], 0)))
    # keys / encryptor / decryptor
    def enc_without(L, o, which):
        e = vp()
        rc = L.rc("Encryptor_Create", L.ctx, o["pk"] if which == "sk" else None, o["sk"] if which == "pk" else None, C.byref(e))
        if rc:
            return ("create", rc)
        name = "Encryptor_Encrypt" if which == "pk" else "Encryptor_EncryptSymmetric"
        args = (e, new_pt(L, [1]), o["dst"], None) if which == "pk" else (e, new_pt(L, [1]), C.c_bool(False), o["dst"], None)
        return ("use", L.rc(name, *args))
    both("Encrypt without a public key", lambda L, o: enc_without(L, o, "pk"))
    both("EncryptSymmetric without a secret key", lambda L, o: enc_without(L, o, "sk"))
    both("Encryptor_Create without any key", lambda L, o: L.rc("Encryptor_Create", L.ctx, None, None, C.byref(vp())))
    def dec_of(L, o, h):
        d = vp()
        L.call("Decryptor_Create", L.ctx, o["sk"], C.byref(d))
        return (L.rc("Decryptor_Decrypt", d, h, o["pt"]), L.rc("Decryptor_InvariantNoiseBudget", d, h, C.byref(C.c_int())))
    both("Decrypt an empty ciphertext", lambda L, o: dec_of(L, o, o["dst"]))
    def ntt_flagged(L, o):
        L.call("Ciphertext_SetIsNTTForm", o["ct"], C.c_bool(True))
        return dec_of(L, o, o["ct"])
    both("Decrypt a ciphertext flagged NTT", ntt_flagged)
    both("Decryptor_Create with a public key handle's parms (wrong object contents)",
         lambda L, o: L.rc("Decryptor_Create", L.ctx, L.load("SecretKey", blob["sk"], unsafe=True), C.byref(vp())))
    both("KeyGenerator_Create2 from a loaded secret key, then relin keys usable",
         lambda L, o: (lambda kg2: (L.rc("KeyGenerator_Create2", L.ctx, o["sk"], C.byref(kg2)), L.rc("KeyGenerator_CreateRelinKeys", kg2, C.c_bool(False), C.byref(vp()))))(vp()))
    # (KSwitchKeys_GetKeyList with an index past the end throws through the reference's C layer and aborts the process:
    #  not comparable)
    if t % (2 * n) == 1:
        def be_case(L, o, vals):
            be = vp()
            L.call("BatchEncoder_Create", L.ctx, C.byref(be))
            arr = (u64 * len(vals))(*vals)
            rc = L.rc("BatchEncoder_Encode1", be, u64(len(vals)), arr, o["pt"])
            return (rc, L.save("Plaintext", o["pt"], 0) if rc == 0 else None)
        def be_signed(L, o, vals):
            be = vp()
            L.call("BatchEncoder_Create", L.ctx, C.byref(be))
            arr = (C.c_int64 * len(vals))(*vals)
            rc = L.rc("BatchEncoder_Encode2", be, u64(len(vals)), arr, o["pt"])
            return (rc, L.save("Plaintext", o["pt"], 0) if rc == 0 else None)
        both("BatchEncoder value == t (the reference checks ranges only in debug builds)", lambda L, o: be_case(L, o, [1, t]))
        both("BatchEncoder signed values beyond +-t/2", lambda L, o: be_signed(L, o, [3, -(t // 2) - 5, t // 2 + 7]))
        both("BatchEncoder too many values", lambda L, o: be_case(L, o, [1] * (n + 1)))
    else:
        both("BatchEncoder_Create without batching", lambda L, o: L.rc("BatchEncoder_Create", L.ctx, C.byref(vp())))
    assert not mismatches, "HRESULT / value mismatches:\\n  " + "\\n  ".join(mismatches)


def context_validation_sweep(S):
    """SEALContext_Create over valid and invalid parameter sets (S/context.cpp:135-420): both libraries agree on
    parameters_set, on key switching / batching support and on the three parms_ids (the reference's answers come from its
    library when present, else from their records: parity_checks.expect)."""
    Rl = refseal.RefLib.get() if refseal.have_ref() else None
    p27 = [0x7e00001, 0x7d20001, 0x7c80001, 0x7b40001]          # 27-bit primes = 1 mod 8192? (checked by the reference)
    d4096, d8192 = [0xffffee001, 0xffffc4001, 0x1ffffe0001], [0x7fffffd8001, 0x7fffffc8001, 0xfffffffc001, 0xffffff6c001, 0xfffffebc001]
    cases = [
        ("default 4096 / TC128", 4096, d4096, 65537, 128, True), ("default 4096 / TC192 (too many bits)", 4096, d4096, 65537, 192, True),
        ("default 4096 / no security", 4096, d4096, 65537, 0, True), ("default 8192, no chain expansion", 8192, d8192, 1032193, 128, False),
        ("default 8192 / TC256 (too many bits)", 8192, d8192, 1032193, 256, True),
        ("8192 chain used at n = 4096 (too many bits)", 4096, d8192, 65537, 128, True), ("same without security", 4096, d8192, 65537, 0, True),
        ("27-bit primes", 4096, p27, 65537, 128, True), ("repeated prime", 4096, [d4096[0], d4096[0], d4096[2]], 65537, 128, True),
        ("composite modulus", 4096, [d4096[0], 0xffffee001 + 2 * 8192, d4096[2]], 65537, 0, True),
        ("modulus not 1 mod 2n", 4096, [d4096[0], 0xffffee003, d4096[2]], 65537, 0, True),
        ("n not a power of two", 3000, d4096, 65537, 0, True), ("n = 512 without security", 512, [0x7e00001], 17, 0, True),
        ("n = 1024 default", 1024, [0x7e00001], 1 << 8, 128, True), ("n = 2048 default", 2048, [0x3fffffff000001], 65537, 128, True),
        ("t = 2 (smallest)", 4096, d4096, 2, 128, True), ("t = 1", 4096, d4096, 1, 128, True), ("t even, no batching", 4096, d4096, 1 << 18, 128, True),
        ("t shares a factor with q", 4096, d4096, d4096[0], 128, True), ("t larger than every q_i", 4096, d4096, 0x1ffffe0001 + 2, 0, True),
        ("t = 1 mod 2n but composite", 4096, d4096, 8193 * 3 if (8193 * 3) % 8192 == 1 else 8192 * 5 + 1, 128, True),
        ("single small prime, t close to q", 1024, [0x7e00001], 0x7e00001 - 2, 0, True), ("61-bit prime", 8192, [0x1fffffffffe00001, 0xfffffffc001], 65537, 0, True),
        ("62-bit modulus", 8192, [0x3fffffffffe00001, 0xfffffffc001], 65537, 0, True), ("no coefficient modulus", 4096, [], 65537, 128, True),
    ]
    mismatches = []
    for label, n, moduli, t, sec, expand in cases:
        def answers(call, rc):
            out = []
            parms = vp()
            call("EncParams_Create1", C.c_uint8(1), C.byref(parms))
            out.append(rc("EncParams_SetPolyModulusDegree", parms, u64(n)))
            arr = (vp * max(len(moduli), 1))()
            ok = True
            for i, m in enumerate(moduli):
                h = vp()
                r = rc("Modulus_Create1", u64(m), C.byref(h))
                out.append(r)
                ok = ok and r == 0
                arr[i] = h
            if ok:
                out.append(rc("EncParams_SetCoeffModulus", parms, u64(len(moduli)), arr))
                out.append(rc("EncParams_SetPlainModulus2", parms, u64(t)))
                ctx = vp()
                r = rc("SEALContext_Create", parms, C.c_bool(expand), C.c_int(sec), C.byref(ctx))
                out.append(r)
                if r == 0:
                    flag = C.c_bool()
                    call("SEALContext_ParametersSet", ctx, C.byref(flag))
                    out.append(flag.value)
                    if flag.value:
                        call("SEALContext_UsingKeyswitching", ctx, C.byref(flag))
                        out.append(flag.value)
                        for name in ("KeyParmsId", "FirstParmsId", "LastParmsId"):
                            a = (u64 * 4)()
                            call("SEALContext_" + name, ctx, a)
                            out.append(tuple(a))
                        be = vp()
                        out.append(rc("BatchEncoder_Create", ctx, C.byref(be)) == 0)
            return json.loads(json.dumps(out))
        res = [expect(f"context validation/{label}", lambda Rl: answers(Rl.call, Rl.call_rc), Rl), answers(S.call, S.rc)]
        if res[0] != res[1]:
            mismatches.append(f"{label}: reference {res[0][-6:]}, ours {res[1][-6:]}")
    assert not mismatches, "context validation differs:\\n  " + "\\n  ".join(mismatches)


def concurrent_evaluator_calls(S, n, moduli, t, threads=8, rounds=6):
    """sunscreen_runtime drives one Evaluator from rayon workers (run.rs:415-469): shared read-only inputs, fresh
    destinations, any interleaving.  Eight Python threads (ctypes drops the GIL in the call) replay that against our library;
    every result must equal the serial one."""
    import threading
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    RL, OL = _libs(R, O)
    kg = R.keygen()
    sk, pk, rlk = R.secret_key(kg), R.public_key(kg), R.relin_keys(kg)
    enc = R.encryptor(pk, sk)
    rng = np.random.default_rng(77)
    cts = [OL.load("Ciphertext", RL.save("Ciphertext", R.encrypt(enc, R.new_pt(rng.integers(0, t, size=16, dtype=np.uint64))), 0)) for _ in range(4)]
    orlk = OL.load("KSwitchKeys", RL.save("KSwitchKeys", rlk, 0))
    pl = O.new_pt(rng.integers(1, t, size=9, dtype=np.uint64))
    batching = t % (2 * n) == 1
    glk = R.galois_keys_steps(kg, [1, 2]) if batching else None
    oglk = OL.load("KSwitchKeys", RL.save("KSwitchKeys", glk, 0)) if batching else None

    def work(i):
        a, b = cts[i % 4], cts[(i + 1) % 4]
        m = O.relinearize(O.multiply(a, b), orlk)
        s = O.add(m, a)
        if batching:  # rotations with a present key go through the combiner too (two different steps -> two batch groups)
            s = O.rotate_rows(s, 1 + (i & 1), oglk)
        p = O.multiply_plain(s, pl)
        return OL.save("Ciphertext", O.sub(p, b), 0)

    serial = [work(i) for i in range(threads)]
    results = [[None] * rounds for _ in range(threads)]
    errors = []

    def runner(i):
        try:
            for r in range(rounds):
                results[i][r] = work(i)
        except Exception as e:  # pragma: no cover
            errors.append((i, repr(e)))

    ts = [threading.Thread(target=runner, args=(i,)) for i in range(threads)]
    for th in ts:
        th.start()
    for th in ts:
        th.join()
    assert not errors, errors
    for i in range(threads):
        for r in range(rounds):
            assert results[i][r] == serial[i], f"thread {i}, round {r}: result differs from the serial evaluation"
    # and the serial results are the reference's
    rcts = [RL.load("Ciphertext", OL.save("Ciphertext", h, 0)) for h in cts]
    rpl = R.new_pt(O.pt_coeffs(pl))
    for i in range(threads):
        a, b = rcts[i % 4], rcts[(i + 1) % 4]
        e1 = R.add(R.relinearize(R.multiply(a, b), rlk), a)
        if batching:
            e1 = R.rotate_rows(e1, 1 + (i & 1), glk)
        exp = R.sub(R.multiply_plain(e1, rpl), b)
        assert RL.save("Ciphertext", exp, 0) == serial[i]


def combined_calls_isolation(S, n, moduli, t, threads=8, rounds=8):
    """Concurrent Evaluator_Multiply / Evaluator_Relinearize calls are run together as one batch by whichever caller holds
    the combiner (sealc_api.cpp: combine_submit).  Each call must still behave as if it ran alone: in-place destinations,
    operands shared between callers, and a caller whose result is transparent (its product with an all-zero ciphertext)
    gets COR_E_INVALIDOPERATION every time while the calls batched with it succeed with the serial words."""
    import threading
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    RL, OL = _libs(R, O)
    kg = R.keygen()
    sk, pk, rlk = R.secret_key(kg), R.public_key(kg), R.relin_keys(kg)
    enc = R.encryptor(pk, sk)
    rng = np.random.default_rng(5)
    rcts = [R.encrypt(enc, R.new_pt(rng.integers(0, t, size=8, dtype=np.uint64))) for _ in range(3)]
    cts = [OL.load("Ciphertext", RL.save("Ciphertext", h, 0)) for h in rcts]
    orlk = OL.load("KSwitchKeys", RL.save("KSwitchKeys", rlk, 0))
    zero = O.new_ct(np.zeros((2, O.k, n), dtype=np.uint64))
    words = lambda h: OL.save("Ciphertext", h, 0)
    expect = {i: RL.save("Ciphertext", R.relinearize(R.multiply(rcts[i % 3], rcts[(i + 1) % 3]), rlk), 0) for i in range(threads)}
    errors, bad = [], []

    def runner(i):
        try:
            for r in range(rounds):
                if i == 0:  # transparent result, every round
                    rc = S.rc("Evaluator_Multiply", O.ev, cts[0], zero, OL.new("Ciphertext"), None)
                    if rc != COR_E_INVALIDOPERATION:
                        bad.append((i, r, hex(rc)))
                    continue
                mine = OL.load("Ciphertext", words(cts[i % 3]))  # private copy, multiplied IN PLACE
                S.call("Evaluator_Multiply", O.ev, mine, cts[(i + 1) % 3], mine, None)
                S.call("Evaluator_Relinearize", O.ev, mine, orlk, mine, None)
                if words(mine) != expect[i]:
                    bad.append((i, r, "words"))
        except Exception as e:  # pragma: no cover
            errors.append((i, repr(e)))

    ts = [threading.Thread(target=runner, args=(i,)) for i in range(threads)]
    for th in ts:
        th.start()
    for th in ts:
        th.join()
    assert not errors, errors
    assert not bad, bad


def handle_lifetime_order(S, n, moduli, t):
    """Rust drops handles in whatever order the program's scopes dictate.  The reference's objects share the context's
    internals, so an Evaluator / Decryptor / ciphertext stays usable after SEALContext_Destroy; ours must too (the device
    context is reference-counted).  The same out-of-order sequence runs against both libraries (the reference's
    serialisations come from its library when present, else from the records of their SHA-256: parity_checks.expect)."""
    import hashlib
    inp = refseal.appendix_b_inputs(n, moduli, t)

    def run(L, ctx, ev, a, b):
        prod = L.new("Ciphertext")
        L.call("Evaluator_Multiply", ev, a, b, prod, None)          # device-resident result
        L.call("SEALContext_Destroy", ctx)                          # the context handle goes first
        s = L.new("Ciphertext")
        L.call("Evaluator_Add", ev, prod, prod, s)                  # the evaluator still works
        words = L.save("Ciphertext", s, 0)
        L.call("Evaluator_Destroy", ev)                             # then the evaluator
        after = L.save("Ciphertext", prod, 0)                       # ciphertexts outlive both
        for h in (a, b, prod, s):
            L.call("Ciphertext_Destroy", h)
        return [hashlib.sha256(words).hexdigest(), hashlib.sha256(after).hexdigest()]

    def ref_run(Rl):
        R = refseal.RefContext(n, moduli, t)
        return run(_Lib(R.ref.call, R.ref.call_rc, R.ctx), R.ctx, R.ev, R.new_ct(inp["a"]), R.new_ct(inp["b"]))
    exp = expect(f"{param_name(n, moduli, t)}/sealc handle lifetime order", ref_run,
                 refseal.RefLib.get() if refseal.have_ref() else None)
    O = S.context(n, moduli, t)
    assert run(_Lib(O.S.call, O.S.rc, O.ctx), O.ctx, O.ev, O.new_ct(inp["a"]), O.new_ct(inp["b"])) == exp


def wire_fuzz(S, n, moduli, t, trials=160, seed=1234):
    """Corrupted and truncated serialisations: our loader never crashes and answers with the reference's HRESULT (and, when both
    accept, holds the same object afterwards)."""
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    RL, OL = _libs(R, O)
    kg = R.keygen()
    sk, pk, rlk = R.secret_key(kg), R.public_key(kg), R.relin_keys(kg)
    ct = R.encrypt(R.encryptor(pk), R.new_pt(np.arange(3, 40, dtype=np.uint64) % t))
    sct = R.new_ct()
    R.ref.call("Encryptor_EncryptSymmetric", R.encryptor(pk, sk), R.new_pt(np.array([5, 6], dtype=np.uint64)), C.c_bool(True), sct, None)
    blobs = [("Ciphertext", RL.save("Ciphertext", ct, 0)), ("Ciphertext", RL.save("Ciphertext", sct, 0)),
             ("Plaintext", RL.save("Plaintext", R.new_pt(np.arange(9, dtype=np.uint64)), 0)), ("SecretKey", RL.save("SecretKey", sk, 0)),
             ("PublicKey", RL.save("PublicKey", pk, 0)), ("KSwitchKeys", RL.save("KSwitchKeys", rlk, 0)),
             ("Ciphertext", RL.save("Ciphertext", ct, COMPR_ZLIB)), ("Ciphertext", RL.save("Ciphertext", ct, COMPR_ZSTD))]
    rng = np.random.default_rng(seed)
    mismatches = []
    for trial in range(trials):
        kind, raw = blobs[trial % len(blobs)]
        data = bytearray(raw)
        mode = trial % 6
        compressed = raw[5] != 0
        if mode == 0:      # one byte in the headers / metadata region
            i = int(rng.integers(0, min(len(data), 140)))
            data[i] ^= int(rng.integers(1, 256))
        elif mode == 1:    # one byte anywhere
            i = int(rng.integers(0, len(data)))
            data[i] ^= 1 << int(rng.integers(0, 8))
        elif mode == 2:    # truncate
            data = data[: int(rng.integers(0, len(data)))]
        elif mode == 3:    # a size / count field set to something else (moderate: the reference allocates what it is told)
            i = int(rng.integers(0, min(len(data) - 8, 140)))
            data[i:i + 8] = int(rng.integers(0, 2**20)).to_bytes(8, "little")
        elif mode == 5:    # ... or to something absurd: the reference dies of an uncaught bad_alloc here, so only OUR loader is
            i = int(rng.integers(0, min(len(data) - 8, 140)))   # asked — it must refuse without allocating
            data[i:i + 8] = int(rng.integers(2**40, 2**63)).to_bytes(8, "little")
            for unsafe in (False, True):
                OL.load_rc(kind, OL.new(kind), bytes(data), unsafe)
            continue
        else:              # trailing garbage after a valid object
            data = data + bytes(rng.integers(0, 256, size=int(rng.integers(1, 64)), dtype=np.uint8))
        data = bytes(data)
        if kind == "KSwitchKeys" and mode in (0, 1, 3) and data[48:64] != raw[48:64]:
            # the two list-length fields: the reference reserves whatever they say and aborts on bad_alloc; ours only
            for unsafe in (False, True):
                OL.load_rc(kind, OL.new(kind), data, unsafe)
            continue
        for unsafe in (False, True):
            rh, oh = RL.new(kind), OL.new(kind)
            r_rc, r_n = RL.load_rc(kind, rh, data, unsafe)
            o_rc, o_n = OL.load_rc(kind, oh, data, unsafe)
            if compressed and mode in (0, 1, 3) and r_rc != 0 and o_rc != 0:
                continue  # both reject a damaged compressed stream; which layer notices first is the compressor's business
            if (r_rc, r_n if r_rc == 0 else 0) != (o_rc, o_n if o_rc == 0 else 0):
                mismatches.append(f"trial {trial} ({kind}, mode {mode}, unsafe={unsafe}): reference 0x{r_rc:08x}/{r_n}, ours 0x{o_rc:08x}/{o_n}")
            elif r_rc == 0 and RL.save(kind, rh, 0) != OL.save(kind, oh, 0):
                mismatches.append(f"trial {trial} ({kind}, mode {mode}): both accept but hold different objects")
    assert not mismatches, "\\n  ".join(["wire fuzz mismatches:"] + mismatches[:12])


def batch_seams(S, n, moduli, t, count=5):
    """B200_Evaluator_{MultiplyRelin,AddSub,Plain,RotateRows}Batch give, item by item, the words of the per-handle calls
    (which the other checks pin to the reference), including in-place destinations and the error cases."""
    R = refseal.RefContext(n, moduli, t)
    O = S.context(n, moduli, t)
    RL, OL = _libs(R, O)
    kg = R.keygen()
    sk, pk, rlk = R.secret_key(kg), R.public_key(kg), R.relin_keys(kg)
    batching = t % (2 * n) == 1
    glk = R.galois_keys_steps(kg, [2]) if batching else None
    enc = R.encryptor(pk)
    rng = np.random.default_rng(41)
    msgs = [rng.integers(0, t, size=int(rng.integers(1, n)), dtype=np.uint64) for _ in range(2 * count)]
    rcts = [R.encrypt(enc, R.new_pt(m)) for m in msgs]
    octs = [OL.load("Ciphertext", RL.save("Ciphertext", h, 0)) for h in rcts]
    A, B = octs[:count], octs[count:]
    orlk = OL.load("KSwitchKeys", RL.save("KSwitchKeys", rlk, 0))
    words = lambda h: OL.save("Ciphertext", h, 0)
    arr = lambda hs: (vp * len(hs))(*hs)
    fresh = lambda: [OL.new("Ciphertext") for _ in range(count)]
    # multiply + relinearize
    d = fresh()
    O.S.call("B200_Evaluator_MultiplyRelinBatch", O.ev, u64(count), arr(A), arr(B), orlk, arr(d))
    for i in range(count):
        assert words(d[i]) == words(O.relinearize(O.multiply(A[i], B[i]), orlk)), f"MultiplyRelinBatch item {i}"
    assert words(d[0]) == RL.save("Ciphertext", R.relinearize(R.multiply(rcts[0], rcts[count]), rlk), 0)
    # add / sub
    for sub in (False, True):
        d = fresh()
        O.S.call("B200_Evaluator_AddSubBatch", O.ev, u64(count), arr(A), arr(B), C.c_bool(sub), arr(d))
        for i in range(count):
            assert words(d[i]) == words((O.sub if sub else O.add)(A[i], B[i])), f"AddSubBatch(sub={sub}) item {i}"
    # plain operations, one plaintext per item
    pls = [rng.integers(1, t, size=int(rng.integers(1, n)), dtype=np.uint64) for _ in range(count)]
    opl = [O.new_pt(p) for p in pls]
    for which, fn in ((0, O.add_plain), (1, O.sub_plain), (2, O.multiply_plain)):
        d = fresh()
        O.S.call("B200_Evaluator_PlainBatch", O.ev, C.c_int(which), u64(count), arr(A), arr(opl), arr(d))
        for i in range(count):
            assert words(d[i]) == words(fn(A[i], opl[i])), f"PlainBatch({which}) item {i}"
    assert S.rc("B200_Evaluator_PlainBatch", O.ev, C.c_int(7), u64(count), arr(A), arr(opl), arr(fresh())) == E_INVALIDARG
    zero = [O.new_pt(np.zeros(3, dtype=np.uint64))] + opl[1:]
    assert S.rc("B200_Evaluator_PlainBatch", O.ev, C.c_int(2), u64(count), arr(A), arr(zero), arr(fresh())) == COR_E_INVALIDOPERATION
    # rotations
    if batching:
        oglk = OL.load("KSwitchKeys", RL.save("KSwitchKeys", glk, 0))
        d = fresh()
        O.S.call("B200_Evaluator_RotateRowsBatch", O.ev, u64(count), arr(A), C.c_int(2), oglk, arr(d))
        for i in range(count):
            assert words(d[i]) == words(O.rotate_rows(A[i], 2, oglk)), f"RotateRowsBatch item {i}"
        assert words(d[1]) == RL.save("Ciphertext", R.rotate_rows(rcts[1], 2, glk), 0)
        assert S.rc("B200_Evaluator_RotateRowsBatch", O.ev, u64(count), arr(A), C.c_int(3), oglk, arr(fresh())) == E_INVALIDARG
    # in place: destinations are the first operands
    mine = [OL.load("Ciphertext", RL.save("Ciphertext", h, 0)) for h in rcts[:count]]
    exp = [words(O.add(A[i], B[i])) for i in range(count)]
    O.S.call("B200_Evaluator_AddSubBatch", O.ev, u64(count), arr(mine), arr(B), C.c_bool(False), arr(mine))
    assert [words(h) for h in mine] == exp
    # items at different levels are rejected
    lower = O.mod_switch_to_next(A[1])
    assert S.rc("B200_Evaluator_AddSubBatch", O.ev, u64(2), arr([A[0], lower]), arr([B[0], B[1]]), C.c_bool(False), arr(fresh()[:2])) == E_INVALIDARG
    # transparent items are reported
    assert S.rc("B200_Evaluator_AddSubBatch", O.ev, u64(2), arr([A[0], A[1]]), arr([B[0], A[1]]), C.c_bool(True), arr(fresh()[:2])) == COR_E_INVALIDOPERATION
    # a null handle anywhere in an argument array, a size-3 item, an NTT-form... : rejected before anything is launched
    holes = (vp * 2)(A[0], None)
    assert S.rc("B200_Evaluator_AddSubBatch", O.ev, u64(2), holes, arr(B[:2]), C.c_bool(False), arr(fresh()[:2])) == E_INVALIDARG
    assert S.rc("B200_Evaluator_MultiplyRelinBatch", O.ev, u64(2), arr(A[:2]), holes, orlk, arr(fresh()[:2])) == E_INVALIDARG
    assert S.rc("B200_Evaluator_MultiplyRelinBatch", O.ev, u64(2), arr(A[:2]), arr(B[:2]), orlk, holes) == E_INVALIDARG
    assert S.rc("B200_Evaluator_MultiplyRelinBatch", O.ev, u64(2), None, arr(B[:2]), orlk, arr(fresh()[:2])) == E_POINTER
    size3 = O.multiply(A[0], B[0])
    assert S.rc("B200_Evaluator_MultiplyRelinBatch", O.ev, u64(2), arr([size3, A[1]]), arr(B[:2]), orlk, arr(fresh()[:2])) == E_INVALIDARG
    assert S.rc("B200_Evaluator_AddSubBatch", O.ev, u64(2), arr([A[0], size3]), arr(B[:2]), C.c_bool(False), arr(fresh()[:2])) == E_INVALIDARG
    if batching:
        assert S.rc("B200_Evaluator_RotateRowsBatch", O.ev, u64(1), arr([size3]), C.c_int(2), oglk, arr(fresh()[:1])) == E_INVALIDARG
    # relinearization keys of another context / an empty key object
    empty = OL.new("KSwitchKeys")
    assert S.rc("B200_Evaluator_MultiplyRelinBatch", O.ev, u64(2), arr(A[:2]), arr(B[:2]), empty, arr(fresh()[:2])) == E_INVALIDARG
    # count == 0 is a no-op
    assert S.rc("B200_Evaluator_MultiplyRelinBatch", O.ev, u64(0), arr(A[:1]), arr(B[:1]), orlk, arr(fresh()[:1])) == 0
    # bulk word access: one contiguous buffer <-> `count` handles
    slab = np.stack([O.ct_words(h) for h in A])                                       # (count, 2, k, n)
    hs = fresh()
    O.S.call("B200_Ciphertext_SetWordsBatch", O.ctx, u64(count), arr(hs), O.first_id, u64(2), C.c_bool(False),
             slab.ctypes.data_as(C.POINTER(u64)))
    for i in range(count):
        assert words(hs[i]) == words(A[i]), f"SetWordsBatch item {i}"
    back = np.zeros_like(slab)
    O.S.call("B200_Ciphertext_GetWordsBatch", O.ctx, u64(count), arr(hs), back.ctypes.data_as(C.POINTER(u64)), u64(back.size))
    eq(back, slab, "GetWordsBatch")
    d = fresh()
    O.S.call("B200_Evaluator_MultiplyRelinBatch", O.ev, u64(count), arr(hs), arr(B), orlk, arr(d))
    O.S.call("B200_Ciphertext_GetWordsBatch", O.ctx, u64(count), arr(d), back.ctypes.data_as(C.POINTER(u64)), u64(back.size))
    eq(back[0], R.ct_words(R.relinearize(R.multiply(rcts[0], rcts[count]), rlk)), "SetWordsBatch -> MultiplyRelinBatch -> GetWordsBatch")
    assert S.rc("B200_Ciphertext_GetWordsBatch", O.ctx, u64(count), arr(d), back.ctypes.data_as(C.POINTER(u64)), u64(back.size - 1)) == E_INVALIDARG
    assert S.rc("B200_Ciphertext_SetWordsBatch", O.ctx, u64(count), arr(hs), O.first_id, u64(1), C.c_bool(False),
                slab.ctypes.data_as(C.POINTER(u64))) == E_INVALIDARG
    assert S.rc("B200_Ciphertext_GetWordsBatch", O.ctx, u64(2), arr([d[0], size3]), back.ctypes.data_as(C.POINTER(u64)), u64(back.size)) == E_INVALIDARG
