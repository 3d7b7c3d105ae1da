"""Word-for-word parity checks of the B200 path against the unmodified reference (shared by CPU-emu and GPU tests).

Every value the reference contributes is also kept in tests/golden/reference_parity.json (arrays as a SHA-256 digest of
their little-endian words, small values as they are), so the checks run without the reference library: with it, each
reference output is compared with the B200 output and with its stored record; without it, the B200 output is compared
with the stored record.  B200_RECORD_GOLDEN=<file> writes the records of a run with the reference to <file>."""
import atexit
import hashlib
import json
import os

import numpy as np

from params import PARAMS
from refseal import RefContext, appendix_b_inputs, have_ref
from sunscreen_b200.lib import B200Context

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_parity.json")
_golden = None
_recorded = {}


def _stored():
    global _golden
    if _golden is None:
        with open(GOLDEN) as f:
            _golden = json.load(f)
    return _golden


def _write_records():
    path = os.environ["B200_RECORD_GOLDEN"]
    old = {}
    if os.path.exists(path):
        with open(path) as f:
            old = json.load(f)
    old.update(_recorded)
    with open(path, "w") as f:
        json.dump(dict(sorted(old.items())), f, indent=0, sort_keys=True)
        f.write("\n")


if os.environ.get("B200_RECORD_GOLDEN"):
    atexit.register(_write_records)


class Digest:
    """A stored reference array: its word count and the SHA-256 of its little-endian uint64 words."""

    def __init__(self, rec):
        self.size, self.sha256 = rec["size"], rec["sha256"]


def _words_sha256(arr):
    return hashlib.sha256(np.ascontiguousarray(arr, dtype="<u8").tobytes()).hexdigest()


def _record(val):
    if isinstance(val, np.ndarray):
        return {"size": int(val.size), "sha256": _words_sha256(val)}
    return json.loads(json.dumps(val))


def param_name(n, moduli, t):
    for name, (pn, pm, pt) in PARAMS.items():
        if (pn, [int(m) for m in pm], pt) == (n, [int(m) for m in moduli], t):
            return name
    raise KeyError(f"no PARAMS entry for n={n}, t={t}")


class Pair:
    """Same parameters instantiated on the B200 library and, when its library is present, on the reference."""

    def __init__(self, be, n, moduli, t):
        self.be = be
        self.n, self.moduli, self.t = n, list(moduli), t
        self.name = param_name(n, moduli, t)
        self.ref = RefContext(n, moduli, t) if have_ref() else None
        self.ctx = B200Context(n, moduli, t, lib=be.lib)
        self.k = self.ctx.k()
        self.inp = appendix_b_inputs(n, self.moduli, t)

    def expect(self, label, fn):
        """The reference's value for `label` on this parameter set (see `expect`)."""
        return expect(f"{self.name}/{label}", fn, self.ref)

    def dev(self, arr):
        return self.be.to_dev(arr)

    def host(self, x):
        return self.be.to_host(x)

    def out(self, *shape):
        return self.be.empty(shape)


def expect(key, fn, ref):
    """The reference's value stored under `key`: fn(ref) when the reference is present (`ref` is not None; checked
    against, or recorded as, the stored record), else the stored record (a Digest for an array)."""
    if ref is not None:
        val = fn(ref)
        rec = _record(val)
        if os.environ.get("B200_RECORD_GOLDEN"):
            _recorded[key] = rec
        else:
            assert _stored().get(key) == rec, f"{key}: the reference's output differs from {GOLDEN}"
        return val
    assert key in _stored(), f"{key}: no stored reference output in {GOLDEN}"
    rec = _stored()[key]
    return Digest(rec) if isinstance(rec, dict) and "sha256" in rec else rec


def rand_ct(rng, moduli, k, n, size=2, batch=None):
    shape = (size, k, n) if batch is None else (batch, size, k, n)
    out = np.empty(shape, dtype=np.uint64)
    for i in range(k):
        out[..., i, :] = rng.integers(0, moduli[i], size=shape[:-2] + (n,), dtype=np.uint64)
    return out


def rand_ksk(rng, moduli, k, n):
    K = len(moduli)
    out = np.empty((k, 2, K, n), dtype=np.uint64)
    for i in range(K):
        out[:, :, i, :] = rng.integers(0, moduli[i], size=(k, 2, n), dtype=np.uint64)
    return out


def eq(got, exp, what):
    if isinstance(exp, Digest):
        got = np.asarray(got).reshape(-1)
        assert got.size == exp.size, f"{what}: {got.size} words vs {exp.size} from the reference"
        assert _words_sha256(got) == exp.sha256, f"{what}: words differ from the reference's (stored digest)"
        return
    got = np.asarray(got).reshape(-1)
    exp = np.asarray(exp).reshape(-1)
    assert got.shape == exp.shape, f"{what}: shape {got.shape} vs {exp.shape}"
    if not np.array_equal(got, exp):
        bad = np.flatnonzero(got != exp)
        raise AssertionError(f"{what}: {bad.size} of {got.size} words differ; first at {bad[:4]}: "
                             f"{got[bad[:4]]} vs {exp[bad[:4]]}")


def check_context(P):
    li = P.ctx.level_info(P.ctx.first_level)
    ri = P.expect("rns_info", lambda R: R.rns_info())
    assert li["parms_id"] == P.expect("first_parms_id", lambda R: list(R.first_parms_id))
    assert P.ctx.level_info(0)["parms_id"] == P.expect("key_parms_id", lambda R: list(R.key_parms_id))
    assert li["gamma"] == ri["gamma"]
    if li["m_sk"] == ri["m_sk"]:
        # the reference's own auxiliary base (61-bit primes)
        assert li["bsk"] == ri["bsk_primes"] and (li["nB"], li["nBsk"]) == (ri["B"], ri["Bsk"])
    else:
        # FP64-friendly auxiliary base: 47..49-bit NTT primes (as wide as the widest user prime), distinct from the user's
        # primes, with at least the reference's dynamic range condition
        # 32 + bits(t) + bits(Q) < bits(prod(B) * m_sk)   (S/util/rns.cpp:617-624); results are base-independent.
        import math
        width = max(47, max(int(m).bit_length() for m in P.moduli))
        assert width <= 49
        assert all(p < (1 << width) and p % (2 * P.n) == 1 for p in li["bsk"]) and len(set(li["bsk"])) == len(li["bsk"])
        assert not set(li["bsk"]) & set(int(m) for m in P.moduli)
        Q = math.prod(li["q"])
        assert math.prod(li["bsk"]).bit_length() > 32 + P.t.bit_length() + Q.bit_length()
    pi = P.expect("plain_info", lambda R: R.plain_info())
    assert li["delta"] == pi["delta"]
    assert li["q_mod_t"] == pi["upper_half_increment"][0] % P.t or li["q_mod_t"] == pi["upper_half_increment"][0]
    assert li["roots"] == P.expect("ntt_roots", lambda R: [R.ref.ntt_root(q, P.n) for q in li["q"]])


def check_ntt(P, items=6, seed=1):
    rng = np.random.default_rng(seed)
    x = rand_ct(rng, P.moduli, P.k, P.n, size=1, batch=items)[:, 0]
    x[0, :, :8] = 0
    x[0, 0, 0] = 1  # delta -> all-ones spectrum
    # magnitude extremes for the lazy (signed FP64 / Harvey) representations: every coefficient q-1, alternating 0 / q-1,
    # and a +-1 pattern (q-1 = -1) that makes the butterflies add up coherently
    qm1 = np.array([m - 1 for m in P.moduli[: P.k]], dtype=np.uint64)[:, None]
    if items >= 6:
        x[3] = np.broadcast_to(qm1, (P.k, P.n))
        x[4] = 0
        x[4, :, ::2] = qm1
        x[5] = 1
        x[5, :, 1::3] = qm1
    d = P.dev(x)
    P.ctx.ntt_forward(d, items)
    got = P.host(d)
    exp = P.expect(f"ntt_forward x{items}", lambda R: np.stack([np.stack([R.ref.ntt_forward(P.moduli[i], x[b, i])
                                                                           for i in range(P.k)]) for b in range(items)]))
    eq(got, exp, "ntt_forward")
    P.ctx.ntt_inverse(d, items)
    eq(P.host(d), x, "ntt round trip")
    # inverse alone of the reference's spectrum (equal to `got`, checked above)
    d2 = P.dev(got)
    P.ctx.ntt_inverse(d2, items)
    eq(P.host(d2), x, "ntt_inverse")


def check_elementwise(P):
    a, b = P.inp["a"], P.inp["b"]
    da, db = P.dev(a), P.dev(b)
    o = P.out(2, P.k, P.n)
    P.ctx.add(da, db, o, 2, 1)
    eq(P.host(o), P.expect("add", lambda R: R.ct_words(R.add(R.new_ct(a), R.new_ct(b)))), "add")
    P.ctx.sub(da, db, o, 2, 1)
    eq(P.host(o), P.expect("sub", lambda R: R.ct_words(R.sub(R.new_ct(a), R.new_ct(b)))), "sub")
    P.ctx.negate(da, o, 2, 1)
    eq(P.host(o), P.expect("negate", lambda R: R.ct_words(R.negate(R.new_ct(a)))), "negate")
    # zero stays zero under negate
    z = np.zeros_like(a)
    P.ctx.negate(P.dev(z), o, 2, 1)
    eq(P.host(o), z, "negate(0)")


def _ref_product(R, P):
    return R.multiply(R.new_ct(P.inp["a"]), R.new_ct(P.inp["b"]))


def check_multiply(P, with_sizes=True):
    """Returns the size-3 product of the App. B operands (equal to the reference's, checked here)."""
    a, b = P.inp["a"], P.inp["b"]
    da, db = P.dev(a), P.dev(b)
    o3 = P.out(3, P.k, P.n)
    P.ctx.multiply(da, 2, db, 2, o3, 1)
    m3 = P.host(o3)
    eq(m3, P.expect("multiply(2,2)", lambda R: R.ct_words(_ref_product(R, P))), "multiply(2,2)")
    P.ctx.square(da, o3, 1)
    eq(P.host(o3), P.expect("square", lambda R: R.ct_words(R.square(R.new_ct(a)))), "square")
    if with_sizes:
        # (3,2) -> 4 : the general K x L convolution loop (S/evaluator.cpp:497-541)
        o4 = P.out(4, P.k, P.n)
        P.ctx.multiply(P.dev(m3), 3, db, 2, o4, 1)
        eq(P.host(o4), P.expect("multiply(3,2)", lambda R: R.ct_words(R.multiply(_ref_product(R, P), R.new_ct(b)))),
           "multiply(3,2)")
    return m3


def check_relin(P, m3):
    exp = P.expect("relinearize", lambda R: R.ct_words(R.relinearize(_ref_product(R, P), R.new_ksk({0: P.inp["rlk"]}))))
    dk = P.dev(P.inp["rlk"])
    o2 = P.out(2, P.k, P.n)
    P.ctx.relinearize(P.dev(m3), dk, o2, 1)
    eq(P.host(o2), exp, "relinearize")
    o2b = P.out(2, P.k, P.n)
    P.ctx.multiply_relin(P.dev(P.inp["a"]), P.dev(P.inp["b"]), dk, o2b, 1)
    eq(P.host(o2b), exp, "multiply_relin")


def check_galois(P):
    n = P.n
    a = P.inp["a"]

    def ref_rotate(step):
        def fn(R):
            glk = R.new_ksk({(3 - 1) // 2: P.inp["glk3"], (2 * n - 1 - 1) // 2: P.inp["glkc"]})
            return R.ct_words(R.rotate_rows(R.new_ct(a), 1, glk) if step else R.rotate_columns(R.new_ct(a), glk))
        return fn
    da = P.dev(a)
    o2 = P.out(2, P.k, P.n)
    assert P.ctx.galois_elt_from_step(1) == 3 and P.ctx.galois_elt_from_step(0) == 2 * n - 1
    P.ctx.apply_galois(da, 3, P.dev(P.inp["glk3"]), o2, 1)
    eq(P.host(o2), P.expect("rotate_rows(1)", ref_rotate(1)), "rotate_rows(1)")
    P.ctx.apply_galois(da, 2 * n - 1, P.dev(P.inp["glkc"]), o2, 1)
    eq(P.host(o2), P.expect("rotate_columns", ref_rotate(0)), "rotate_columns")


def check_plain(P):
    a, p = P.inp["a"], P.inp["p"]
    da, dp = P.dev(a), P.dev(p)
    o2 = P.out(2, P.k, P.n)
    for op in ("multiply_plain", "add_plain", "sub_plain"):
        getattr(P.ctx, op)(da, 2, dp, 1, o2, 1)
        eq(P.host(o2), P.expect(op, lambda R: R.ct_words(getattr(R, op)(R.new_ct(a), R.new_pt(p)))), op)
    # monomial plaintext (the reference takes its fast path, S/evaluator.cpp:1885-1933): same words expected
    mono = np.zeros(P.n, dtype=np.uint64)
    mono[5] = 7
    P.ctx.multiply_plain(da, 2, P.dev(mono), 1, o2, 1)
    eq(P.host(o2), P.expect("multiply_plain(monomial)", lambda R: R.ct_words(R.multiply_plain(R.new_ct(a), R.new_pt(mono[:6])))),
       "multiply_plain(monomial)")


def check_modswitch(P):
    a = P.inp["a"]
    if P.k < 2:
        return
    o = P.out(2, P.k - 1, P.n)
    P.ctx.mod_switch_to_next(P.dev(a), 2, o, 1)
    eq(P.host(o), P.expect("mod_switch_to_next", lambda R: R.ct_words(R.mod_switch_to_next(R.new_ct(a)))), "mod_switch_to_next")


def check_batch(P, batch=3, seed=7):
    """Distinct items in one launch: strides / item indexing."""
    rng = np.random.default_rng(seed)
    A = rand_ct(rng, P.moduli, P.k, P.n, batch=batch)
    B = rand_ct(rng, P.moduli, P.k, P.n, batch=batch)
    key = rand_ksk(rng, P.moduli, P.k, P.n)
    dA, dB, dK = P.dev(A), P.dev(B), P.dev(key)
    o2 = P.out(batch, 2, P.k, P.n)
    o3 = P.out(batch, 3, P.k, P.n)
    P.ctx.multiply(dA, 2, dB, 2, o3, batch)
    got3 = P.host(o3)
    P.ctx.multiply_relin(dA, dB, dK, o2, batch)
    got2 = P.host(o2)
    og = P.out(batch, 2, P.k, P.n)
    P.ctx.apply_galois(dA, 3, dK, og, batch)
    gotg = P.host(og)

    def ref_item(i, op):
        def fn(R):
            ra, rb = R.new_ct(A[i]), R.new_ct(B[i])
            if op == "rotate":
                out = R.rotate_rows(ra, 1, R.new_ksk({1: key}))
            else:
                out = R.multiply(ra, rb)
                if op == "multiply_relin":
                    out = R.relinearize(out, R.new_ksk({0: key}))
            words = R.ct_words(out)
            for h in (ra, rb, out):
                R.free_ct(h)
            return words
        return fn
    for i in range(batch):
        tag = f"item {i} of {batch}, seed {seed}"
        eq(got3[i], P.expect(f"batch multiply {tag}", ref_item(i, "multiply")), f"batch multiply item {i}")
        eq(got2[i], P.expect(f"batch multiply_relin {tag}", ref_item(i, "multiply_relin")), f"batch multiply_relin item {i}")
        if P.ctx.using_batching:
            eq(gotg[i], P.expect(f"batch rotate {tag}", ref_item(i, "rotate")), f"batch rotate item {i}")


def check_encrypted_roundtrip(P, seed=3):
    """Real keys + fresh encryptions from the reference; B200 multiply+relin output decrypts (on the reference
    AND through b200_decrypt) to the slot-wise product, and equals the reference's ciphertext word for word."""
    if P.ref is None:
        import pytest
        pytest.skip("needs the reference library: its keys and encryptions are random, so no stored output stands for them")
    rng = np.random.default_rng(seed)
    R = P.ref
    kg = R.keygen()
    sk, pk, rk = R.secret_key(kg), R.public_key(kg), R.relin_keys(kg)
    enc, dec = R.encryptor(pk), R.decryptor(sk)
    be_ = R.batch_encoder()
    v1 = rng.integers(0, P.t, size=P.n, dtype=np.uint64)
    v2 = rng.integers(0, P.t, size=P.n, dtype=np.uint64)
    c1, c2 = R.encrypt(enc, R.batch_encode(be_, v1)), R.encrypt(enc, R.batch_encode(be_, v2))
    w1, w2 = R.ct_words(c1), R.ct_words(c2)
    key = R.ksk_words(rk)[0]
    exp_ct = R.relinearize(R.multiply(c1, c2), rk)
    o2 = P.out(2, P.k, P.n)
    P.ctx.multiply_relin(P.dev(w1), P.dev(w2), P.dev(key), o2, 1)
    got = P.host(o2)
    eq(got, R.ct_words(exp_ct), "multiply_relin on real ciphertexts")
    back = R.new_ct(got.reshape(2, P.k, P.n))
    assert R.noise_budget(dec, back) > 0
    vals = R.batch_decode(be_, R.decrypt(dec, back))
    expect = (v1.astype(object) * v2.astype(object)) % P.t
    assert np.array_equal(vals.astype(object), expect)
    return dict(dec=dec, sk=sk, ct=got, expect_plain=R.pt_coeffs(R.decrypt(dec, back)))


def check_small_kernels(P, seed=29):
    """b200_is_transparent / b200_any_nonzero (the transparent-result guard, S/ciphertext.h:451-456) on a batch with one
    transparent item and one whose only nonzero word is the very last; b200_expand_signed (residues of the host-sampled
    ternary / clipped-normal values, S/util/rlwe.cpp:23-67) against v mod q_i."""
    rng = np.random.default_rng(seed)
    batch = 4
    ct = rand_ct(rng, P.moduli, P.k, P.n, batch=batch)
    ct[1, 1:] = 0                      # transparent: c1 == 0 (c0 arbitrary)
    ct[2, 1:] = 0
    ct[2, 1, P.k - 1, P.n - 1] = 1     # a single nonzero word at the very end
    d = P.dev(ct)
    words = (batch + 1) // 2
    flags = P.dev(np.zeros(words, dtype=np.uint64))
    P.ctx.is_transparent(d, 2, flags, batch)
    got = P.host(flags).view(np.uint32)[:batch]
    assert list(got) == [0, 1, 0, 0], f"is_transparent flags {list(got)}"
    flags = P.dev(np.zeros(words, dtype=np.uint64))
    P.ctx.any_nonzero(d, 2, flags, batch)
    got = P.host(flags).view(np.uint32)[:batch]
    assert list(got) == [1, 0, 1, 1], f"any_nonzero flags {list(got)}"
    vals = rng.integers(-19, 20, size=(3, P.n), dtype=np.int64)
    vals[0, :4] = (-1, 0, 1, -19)
    out = P.out(3, P.k, P.n)
    P.ctx.expand_signed(P.dev(vals.view(np.uint64)), 3, out)
    got = P.host(out).reshape(3, P.k, P.n)
    for i in range(P.k):
        want = (vals.astype(object) % int(P.moduli[i])).astype(np.uint64)
        eq(got[:, i, :], want, f"expand_signed residue {i}")


def check_noise_norm(P, batch=3, seed=23):
    """b200_noise_norm (the quantity behind invariant_noise_budget, S/decryptor.cpp:424-485): for random ciphertexts of
    size 2 and 3 and random key powers, the device's multi-precision infinity norm of the centred t * phase mod Q equals
    the same computed with Python integers from the phase words."""
    from functools import reduce
    rng = np.random.default_rng(seed)
    q = [int(m) for m in P.moduli[: P.k]]
    Q = reduce(lambda a, b: a * b, q)
    words = (Q.bit_length() + 63) // 64 + 1
    for size in (2, 3):
        ct = rand_ct(rng, P.moduli, P.k, P.n, size=size, batch=batch)
        skp = np.stack([np.stack([rng.integers(0, q[i], size=P.n, dtype=np.uint64) for i in range(P.k)]) for _ in range(size - 1)])
        dct, dsk = P.dev(ct), P.dev(skp)
        ph = P.out(batch, P.k, P.n)
        P.ctx.ct_sk_phase(dct, size, dsk, ph, batch)
        phase = P.host(ph).reshape(batch, P.k, P.n)
        got = np.zeros((batch, words), dtype=np.uint64)
        P.ctx.noise_norm(dct, size, dsk, got, words, batch)
        coef = [(Q // qi) * pow(Q // qi, -1, qi) * P.t % Q for qi in q]
        for b in range(batch):
            best = 0
            for c in range(P.n):
                v = sum(int(phase[b, i, c]) * coef[i] for i in range(P.k)) % Q
                v = Q - v if v >= (Q + 1) // 2 else v
                best = max(best, v)
            mine = sum(int(got[b, w]) << (64 * w) for w in range(words))
            assert mine == best, f"noise norm, size {size}, item {b}: {mine:#x} != {best:#x}"


def check_host_pipeline(P, batch=5, seed=17):
    """b200_multiply_relin_host (host buffers in, host buffers out; chunked, overlapped, packed 6-byte transfers when the
    level's primes fit 48 bits) returns the same words as the device-resident entry point, also when the ring of staging
    slots wraps (chunk of 1 item, 5 items, 3 slots); a word that does not fit the residue width is rejected."""
    import os
    rng = np.random.default_rng(seed)
    A = rand_ct(rng, P.moduli, P.k, P.n, batch=batch)
    B = rand_ct(rng, P.moduli, P.k, P.n, batch=batch)
    key = rand_ksk(rng, P.moduli, P.k, P.n)
    dK = P.dev(key)
    o2 = P.out(batch, 2, P.k, P.n)
    P.ctx.multiply_relin(P.dev(A), P.dev(B), dK, o2, batch)
    want = P.host(o2)
    old = os.environ.get("B200_HOST_CHUNK")
    old_pack = os.environ.get("B200_HOST_PACK")
    try:
        for pack in ("0", "1"):
            os.environ["B200_HOST_PACK"] = pack
            for chunk in ("1", "2", "64"):
                os.environ["B200_HOST_CHUNK"] = chunk
                oh = np.zeros((batch, 2, P.k, P.n), dtype=np.uint64)
                P.ctx.multiply_relin_host(A, B, dK, oh, batch)
                eq(oh, want, f"multiply_relin_host, chunk {chunk}, pack {pack}")
        if max(P.moduli[: P.k]) < 2**48:
            bad = A.copy()
            bad[batch - 1, 1, P.k - 1, P.n - 1] = np.uint64(2**48)
            try:
                P.ctx.multiply_relin_host(bad, B, dK, np.zeros_like(want), batch)
            except Exception as e:  # B200Error(B200_E_INVALID)
                assert "residue width" in str(e) or "-1" in str(e), e
            else:
                raise AssertionError("an out-of-range ciphertext word must be rejected by the packed pipeline")
    finally:
        for name, val in (("B200_HOST_CHUNK", old), ("B200_HOST_PACK", old_pack)):
            if val is None:
                os.environ.pop(name, None)
            else:
                os.environ[name] = val


# ---------------------------------------------------------------------------------------------------------
# adversarial operands: the extremes of every lazy range (signed FP64 values up to 2^53, Harvey [0, 4q), the substituted
# 47..49-bit auxiliary base of the FP64 BEHZ path) — all q-1, alternating 0 / q-1, a +-1 pattern, a single nonzero word
# ---------------------------------------------------------------------------------------------------------
ADVERSARIAL = ("qm1", "alt", "pm1", "single", "one")


def adversarial_ct(P, kind, size=2):
    q = np.array([int(m) for m in P.moduli[: P.k]], dtype=np.uint64)[None, :, None]
    x = np.zeros((size, P.k, P.n), dtype=np.uint64)
    if kind == "qm1":
        x[:] = q - np.uint64(1)
    elif kind == "alt":
        x[:, :, ::2] = np.broadcast_to(q - np.uint64(1), (size, P.k, (P.n + 1) // 2))
    elif kind == "pm1":
        x[:] = 1
        x[:, :, 1::3] = np.broadcast_to(q - np.uint64(1), x[:, :, 1::3].shape)
    elif kind == "single":
        x[:, :, P.n - 1] = np.broadcast_to((q - np.uint64(1))[:, :, 0], (size, P.k))
    elif kind == "one":
        x[:, :, 0] = 1
    else:
        raise ValueError(kind)
    return x


def check_adversarial_multiply(P, pairs=None, with_size5=True):
    """multiply / square / multiply_relin of adversarial operands, word for word against the reference (which runs its own
    61-bit auxiliary base and integer arithmetic throughout)."""
    dk = P.dev(P.inp["rlk"])

    def ref_words(a, b, op):
        def fn(R):
            ra, rb = R.new_ct(a), R.new_ct(b)
            if op == "square":
                out = R.square(ra)
            else:
                out = R.multiply(ra, rb)
                if op == "multiply_relin":
                    out = R.relinearize(out, R.new_ksk({0: P.inp["rlk"]}))
            words = R.ct_words(out)
            for h in (ra, rb, out):
                R.free_ct(h)
            return words
        return fn
    pairs = pairs or [("qm1", "qm1"), ("qm1", "alt"), ("alt", "pm1"), ("pm1", "pm1"), ("single", "qm1"), ("single", "single"),
                      ("one", "qm1"), ("alt", "alt")]
    for ka, kb in pairs:
        a, b = adversarial_ct(P, ka), adversarial_ct(P, kb)
        da, db = P.dev(a), P.dev(b)
        o3 = P.out(3, P.k, P.n)
        P.ctx.multiply(da, 2, db, 2, o3, 1)
        eq(P.host(o3), P.expect(f"multiply({ka},{kb})", ref_words(a, b, "multiply")), f"multiply({ka},{kb})")
        o2 = P.out(2, P.k, P.n)
        P.ctx.multiply_relin(da, db, dk, o2, 1)
        eq(P.host(o2), P.expect(f"multiply_relin({ka},{kb})", ref_words(a, b, "multiply_relin")), f"multiply_relin({ka},{kb})")
        if ka == kb:
            P.ctx.square(da, o3, 1)
            eq(P.host(o3), P.expect(f"square({ka})", ref_words(a, b, "square")), f"square({ka})")
    if with_size5:
        for kind in ("qm1", "alt"):
            a3, b3 = adversarial_ct(P, kind, 3), adversarial_ct(P, "pm1" if kind == "alt" else "qm1", 3)
            o5 = P.out(5, P.k, P.n)
            P.ctx.multiply(P.dev(a3), 3, P.dev(b3), 3, o5, 1)
            label = f"multiply (3,3) -> 5 of {kind}"
            eq(P.host(o5), P.expect(label, ref_words(a3, b3, "multiply")), label)


def check_adversarial_keyswitch(P):
    """relinearize / rotate on adversarial targets with an all-(p-1) key: the key-switch accumulators at their largest."""
    K = len(P.moduli)
    key = np.empty((P.k, 2, K, P.n), dtype=np.uint64)
    for i in range(K):
        key[:, :, i, :] = np.uint64(int(P.moduli[i]) - 1)
    dk = P.dev(key)
    for kind in ("qm1", "alt", "single"):
        m3 = adversarial_ct(P, kind, 3)
        o2 = P.out(2, P.k, P.n)
        P.ctx.relinearize(P.dev(m3), dk, o2, 1)
        label = f"relinearize({kind}) with an all-(p-1) key"
        eq(P.host(o2), P.expect(label, lambda R: R.ct_words(R.relinearize(R.new_ct(m3), R.new_ksk({0: key})))), label)
    if P.ctx.using_batching:
        a = adversarial_ct(P, "qm1")
        o2 = P.out(2, P.k, P.n)
        P.ctx.apply_galois(P.dev(a), 3, dk, o2, 1)
        label = "rotate_rows(qm1) with an all-(p-1) key"
        eq(P.host(o2), P.expect(label, lambda R: R.ct_words(R.rotate_rows(R.new_ct(a), 1, R.new_ksk({1: key})))), label)
