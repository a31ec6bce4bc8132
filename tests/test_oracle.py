"""Pins the oracles: the Python big-int oracle and the C restatement against the golden vectors
(reference outputs for secp256k1, public constants for BN254) and against each other."""
import ctypes as C
import hashlib
import os
import random

import pytest

from oracle import curves_py as O
from oracle import loader
from tests.common import be, bn254_points, det_scalar, enc_points, golden, le, secp_chain

BN, SE = O.BN254, O.SECP256K1


def test_curve_constants():
    for c in (BN, SE):
        G = (c.gx, c.gy)
        assert O.on_curve(c, G)
        assert O.mul(c, c.n, G) is None
        assert O.mul(c, c.n - 1, G) == O.neg(c, G)
    g = golden("bn254.json")
    assert O.bn254_marshal(O.mul(BN, 2, (1, 2))).hex() == g["two_g"]
    # SURVEY.md 8(c): Marshal([tau]G) for Porla's TAU_KEY (config.hpp:39)
    assert g["tau_g"] == ("24070ec18ee42497a55ff81f16429ab97e60ccccf6e82595a0c491f317628d35"
                          "0504cdd69ed930f3268f85b8326573114e58750afa2892af9aba2a53e310c654")
    assert O.bn254_marshal(O.mul(BN, 0xffeeddccbbaa99887766554433221100, (1, 2))).hex() == g["tau_g"]


def test_python_msm_matches_naive():
    rnd = random.Random(2)
    for c in (BN, SE):
        pts = [O.hash_point(c, i) for i in range(12)] + [None]
        sc = [rnd.randrange(1 << 256) for _ in pts]
        assert O.msm(c, sc, pts) == O.msm_naive(c, sc, pts)


def test_python_secp_matches_reference_golden():
    """Python oracle == outputs of the reference's secp256k1_ecmult_multi_var (fixtures)."""
    g = golden("secp256k1_ref.json")
    pts = secp_chain(766)
    for case in g["cases"]:
        n = case["n"]
        if n > 766:
            continue
        sc = [det_scalar(b"porla-sc", i) for i in range(n)]
        r = O.msm(SE, sc, pts[:n])
        assert O.secp_sec1_compressed(r).hex() == case["sec1"], n
        assert (be(r[0]) + be(r[1])).hex() == case["xy"], n
    e = g["edge"]
    n = e["n"]
    sb, pb = bytes.fromhex(e["scalars"]), bytes.fromhex(e["points"])
    sc = [int.from_bytes(sb[32 * i:32 * i + 32], "little") for i in range(n)]
    pts = []
    for i in range(n):
        b = pb[64 * i:64 * i + 64]
        pts.append(None if b == bytes(64) else (int.from_bytes(b[:32], "big"), int.from_bytes(b[32:], "big")))
    assert O.secp_sec1_compressed(O.msm_naive(SE, sc, pts)).hex() == e["sec1"]


def test_python_secp_known_answer_hash():
    """tests.c:4715-4757 (test_ecmult_constants): SHA-256 over the serialisations of x*G for
    74 + 32768 scalars, expected e4711b4d...859ab7b4 (tests.c:4732-4737), recomputed with the
    Python oracle (incremental affine additions keep it fast)."""
    c = SE
    G = (c.gx, c.gy)
    h = hashlib.sha256()

    def put(P):
        h.update(b"\x00" if P is None else O.secp_sec1_uncompressed(P))

    for i in range(37):
        P = O.mul(c, i, G)
        put(P)
        put(O.neg(c, P))
    base = G
    for i in range(256):
        two = O.add(c, base, base)
        cur = base
        for j in range(1, 256, 2):
            put(cur)                      # j * 2^i * G
            cur = O.add(c, cur, two)
        base = two
    assert h.hexdigest() == golden("secp256k1_ref.json")["kat"]["sha256"]


def test_c_oracle_matches_python_and_golden():
    g = golden("bn254.json")
    pts = bn254_points(766)
    assert hashlib.sha256(enc_points(pts)).hexdigest() == g["points_sha256"]
    for case in g["cases"]:
        n = case["n"]
        if case["kind"] == "uniform256":
            sc = [det_scalar(b"porla-sc", i) for i in range(n)]
        else:
            sc = [det_scalar(b"porla-31", i) & 0x7FFFFFFF for i in range(n)]
        got = loader.bn254_msm(b"".join(map(be, sc)), enc_points(pts[:n]), n, 1 if n < 128 else 4)
        assert got.hex() == case["marshal"], (n, case["kind"])


def test_c_oracle_edge_cases():
    rnd = random.Random(9)
    P, Q = bn254_points(2)
    cases = [
        ([5, 5], [P, O.neg(BN, P)]),
        ([3, 4, 9], [P, P, P]),
        ([7, 7, 7, 7], [P, P, Q, Q]),
        ([0, 0], [P, Q]),
        ([BN.n, BN.n + 1], [P, Q]),
        ([BN.n - 1, 1], [P, P]),
        ([(1 << 256) - 1], [Q]),
        ([77], [None]),
    ]
    for sc, pts in cases:
        got = loader.bn254_msm(b"".join(map(be, sc)), enc_points(pts), len(sc))
        assert got == O.bn254_marshal(O.msm_naive(BN, sc, pts)), sc
    assert loader.bn254_msm(b"", b"", 0) == bytes(64)
    lib = loader.bn254()
    out = C.create_string_buffer(64)
    k = rnd.randrange(1 << 256)
    lib.oracle_bn254_mul(O.bn254_marshal(P), be(k), out)
    assert out.raw == O.bn254_marshal(O.mul(BN, k, P))
    lib.oracle_bn254_add(O.bn254_marshal(P), O.bn254_marshal(P), out)
    assert out.raw == O.bn254_marshal(O.add(BN, P, P))


@pytest.mark.skipif(loader.secp_ref() is None, reason="oracle/_ref/libsecp_ref.so not built (needs /root/reference)")
def test_reference_build_reproduces_its_own_golden():
    """oracle/_ref (the unmodified vendored C) reproduces tests.c's known-answer hash and the
    committed fixtures, and has the struct sizes the adapter mirrors (SURVEY.md Appendix D)."""
    lib = loader.secp_ref()
    g = golden("secp256k1_ref.json")
    out = C.create_string_buffer(32)
    assert lib.ref_secp_kat(out, None) == g["kat"]["count"]
    assert out.raw.hex() == g["kat"]["sha256"]
    assert (lib.ref_secp_sizeof_ge(), lib.ref_secp_sizeof_gej(), lib.ref_secp_sizeof_scalar()) == (88, 128, 32)
    n = 128
    chain = C.create_string_buffer(64 * n)
    lib.ref_secp_point_chain(hashlib.sha256(b"porla-seed").digest()[::-1], n, chain)
    assert chain.raw == enc_points(secp_chain(n))
    sc = b"".join(le(det_scalar(b"porla-sc", i)) for i in range(n))
    ok, xy, sec1 = loader.secp_ref_msm(sc, chain.raw, n)
    case = [c for c in g["cases"] if c["n"] == n][0]
    assert ok == 1 and sec1.hex() == case["sec1"]
    # threads = the reference's own range partition (Client.hpp:747-787)
    h = lib.ref_secp_prepare(sc, chain.raw, n)
    o33 = C.create_string_buffer(33)
    assert lib.ref_secp_msm_prepared(h, n, 8, None, o33) == 1 and o33.raw.hex() == case["sec1"]
    lib.ref_secp_release(h)


def test_glv_constants_in_the_kernel_header_and_split_bounds():
    """Bn254::glv_* in porla_b200/csrc/ec.cuh against an independent derivation (cube roots of unity, extended
    Euclid on (r, lambda)), and the size bound of the split the recoder relies on (|k1|, |k2| < 2^127)."""
    import os
    import random
    import re
    from oracle import curves_py as O
    c = O.BN254
    g = O.glv_constants(c)
    assert pow(g["beta"], 3, c.p) == 1 and g["beta"] != 1 and pow(g["lambda"], 3, c.n) == 1 and g["lambda"] != 1
    P = O.hash_point(c, 7)
    assert O.mul(c, g["lambda"], P) == (g["beta"] * P[0] % c.p, P[1])
    assert (g["a1"] + g["b1"] * g["lambda"]) % c.n == 0 and (g["a2"] + g["b2"] * g["lambda"]) % c.n == 0
    assert g["a1"] * g["b2"] - g["a2"] * g["b1"] == c.n and g["b2"] == g["a1"] and g["b1"] < 0
    src = open(os.path.join(os.path.dirname(__file__), "..", "porla_b200", "csrc", "ec.cuh")).read()

    def limbs(name):
        body = re.search(r"%s\(int i\) \{[^}]*?m\[\d+\] = \{([^}]*)\}" % name, src, re.S).group(1)
        return sum(int(tok.strip().rstrip("u"), 16) << (32 * i) for i, tok in enumerate(body.split(",")))

    assert limbs("glv_beta_mont") == g["beta"] * (1 << 256) % c.p
    assert limbs("glv_g1") == (g["b2"] << 256) // c.n
    assert limbs("glv_g2") == ((-g["b1"]) << 256) // c.n
    assert limbs("glv_a1") == g["a1"] and limbs("glv_a2") == g["a2"] and limbs("glv_nb1") == -g["b1"]
    rnd = random.Random(127)
    lam = g["lambda"]
    ks = [0, 1, 2, c.n - 1, c.n - 2, c.n // 2, c.n // 2 + 1, lam, c.n - lam, lam - 1, lam + 1, (1 << 253) % c.n, (1 << 253) - 1,
          1 << 128, (1 << 128) - 1, 1 << 127, g["a2"], g["a2"] - 1, c.n - g["a2"], -g["b1"], c.n + g["b1"]]
    ks += [rnd.randrange(c.n) for _ in range(300000)]
    for k in ks:
        k1, k2 = O.glv_split(c, k, g)
        assert (k1 + k2 * lam - k) % c.n == 0
        assert abs(k1) < 1 << 127 and abs(k2) < 1 << 127


def test_recoding_restatement_on_its_edge_families():
    """oracle/recoding_py.py is the specification the radix-route GPU tests check the window sums against: its digits must
    rebuild s mod the order (k1 + k2 lambda with GLV), stay within 2^(c-1), never carry out of the top window, and come in
    as many windows as porla_msm_plan (host-only) reports, for every window size on both curves, on the families that sit
    on the recoding's edges."""
    import ctypes as C
    import porla_b200 as pb
    from oracle import recoding_py as R
    lam = R.glv_consts()["lambda"]
    lib = pb.load()
    for curve, cv, glv in ((pb.CURVE_BN254, BN, False), (pb.CURVE_BN254, BN, True), (pb.CURVE_SECP256K1, SE, False)):
        signs = set()
        for c in range(2, 25):
            code = c | (pb.lib.PLAN_GLV_ON if glv else pb.lib.PLAN_GLV_OFF)
            got, nwin = C.c_int(0), C.c_int(0)
            lib.porla_msm_plan(curve, (1 << 19) + 37, 1, code, C.byref(got), C.byref(nwin))
            assert got.value == code and nwin.value == R.num_windows(cv, glv, c), (cv.name, glv, c)
            half = 1 << (c - 1)
            for name, vals in R.families(cv, glv, c, 24, seed=c).items():
                for s in vals:
                    parts = R.recode(cv, glv, c, s)
                    total = 0
                    for h, ((sign, digits, carry), (_, mag)) in enumerate(zip(parts, R.halves(cv, glv, s))):
                        where = (cv.name, glv, c, name, hex(s), h)
                        assert len(digits) == nwin.value and carry == 0, where
                        assert all(abs(d) <= half for d in digits), where
                        assert sum(d << (c * w) for w, d in enumerate(digits)) == mag, where
                        if mag and name == "tie":
                            assert digits[0] == half, where
                        if mag and name == "carry_chain":
                            assert digits[0] < 0, where
                        total += sign * (lam if h else 1) * mag
                        signs.add((h, sign, mag == 0))
                    assert (total - s) % cv.n == 0, (cv.name, glv, c, name, hex(s))
                    deltas = R.window_multipliers(cv, glv, c, s)
                    assert (sum(d << (c * w) for w, d in enumerate(deltas)) - s) % cv.n == 0, (cv.name, glv, c, name, hex(s))
        # the families reach the sign cases the kernels handle: the secp256k1 flip, and k2 < 0 and k2 = 0 with GLV
        if cv is SE:
            assert {(0, -1, False), (0, 1, False)} <= signs
        if glv:
            assert {(1, -1, False), (1, 1, True)} <= signs


def test_ipa_transcript_sha_matches_the_reference_object():
    """Porla's IPA prover keeps ONE secp256k1_sha256 and finalizes it again and again (Server.hpp:2306-2310, 2386-2387):
    the oracle's restatement of that object against the reference's own hash_impl.h compiled into oracle/_ref."""
    import random
    import pytest
    from oracle import ipa_py, loader
    rnd = random.Random(2306)
    segs = [bytes(rnd.getrandbits(8) for _ in range(ln)) for ln in (64, 33, 33, 0, 1, 55, 56, 63, 64, 65, 119, 120, 200, 33, 33)]
    ref = loader.secp_ref_sha256_sequence(segs)
    if ref is None:
        pytest.skip("oracle/_ref not built (reference tree absent)")
    t = ipa_py.TranscriptSha256()
    for s, want in zip(segs, ref):
        t.write(s)
        assert t.finalize() == want
    import hashlib
    assert ref[0] == hashlib.sha256(segs[0]).digest() and ref[1] != hashlib.sha256(segs[1]).digest()


def test_ipa_oracle_prover_and_verifier_close_the_loop():
    """The restatements of Server::inner_product_prove (Server.hpp:2279-2443) and Client::inner_product_verify
    (Client.hpp:1465-1630) are two different algebraic statements of the same protocol: a proof of the first must satisfy
    the point equation of the second, and a flipped bit must not."""
    import random
    from oracle import curves_py as O, ipa_py
    c = O.SECP256K1
    rnd = random.Random(1465)
    G = (c.gx, c.gy)
    for n in (4, 16):
        gens = [O.mul(c, rnd.randrange(1, c.n), G) for _ in range(n)]
        u = O.mul(c, rnd.randrange(1, c.n), G)
        a = [rnd.randrange(1 << 256) for _ in range(n)]
        b = [rnd.randrange(c.n) for _ in range(n)]
        proof = ipa_py.inner_product_prove(gens, u, a, b)
        assert len(proof) == 32 + 66 * (n.bit_length() - 2) + 128
        commitment = O.msm(c, [x % c.n for x in a], gens)
        assert ipa_py.inner_product_verify(gens, u, commitment, proof)
        for flip in (0, 35, len(proof) - 1):
            bad = bytearray(proof)
            bad[flip] ^= 1
            assert not ipa_py.inner_product_verify(gens, u, commitment, bytes(bad))
