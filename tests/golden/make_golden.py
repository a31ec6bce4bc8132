"""Generates tests/golden/*.json.  Run in the build container (needs /root/reference for the
secp256k1 vectors: they are OUTPUTS OF THE REFERENCE's own secp256k1_ecmult_multi_var, built
unmodified into oracle/_ref/libsecp_ref.so).  BN254 vectors come from the independent big-int
oracle (gnark-crypto is unavailable: "vs restatement") plus the public constants of SURVEY.md 8(c).

    python tests/golden/make_golden.py
"""
import ctypes as C
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import curves_py as O  # noqa: E402
from oracle import loader  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def det_scalar(tag: bytes, i: int) -> int:
    return int.from_bytes(hashlib.sha256(tag + i.to_bytes(8, "little")).digest(), "big")


def secp_vectors():
    lib = loader.secp_ref()
    assert lib is not None, "needs /root/reference"
    out = {"source": "secp256k1_ecmult_multi_var of /root/reference/porla/Utils/secp256k1_lib (ecmult_impl.h:814), "
                     "zero G-scalar, scratch sized as Client.hpp:755-758",
           "inputs": "points: ref_secp_point_chain(q = sha256('porla-seed'), n) i.e. P0 = G, P(i+1) = P(i) + q*G; "
                     "scalars: sha256('porla-sc' || LE64(i)) as a 256-bit integer, NOT reduced, stored as 32 LE bytes",
           "cases": []}
    q = hashlib.sha256(b"porla-seed").digest()[::-1]
    nmax = 4096
    chain = C.create_string_buffer(64 * nmax)
    lib.ref_secp_point_chain(q, nmax, chain)
    out["chain_sha256"] = hashlib.sha256(chain.raw).hexdigest()
    for n in (1, 2, 3, 16, 87, 88, 96, 128, 766, 4096):
        sc = b"".join(det_scalar(b"porla-sc", i).to_bytes(32, "little") for i in range(n))
        ok, xy, sec1 = loader.secp_ref_msm(sc, chain.raw[: 64 * n], n)
        assert ok == 1
        out["cases"].append({"n": n, "sec1": sec1.hex(), "xy": xy.hex()})
    # edge cases of tests.c:3816-4053 in spirit: infinity inputs, zero scalars, cancelling pair
    n = 8
    pts = bytearray(chain.raw[: 64 * n])
    pts[64 * 2: 64 * 3] = bytes(64)                       # infinity
    p = O.SECP256K1.p
    y3 = int.from_bytes(pts[64 * 3 + 32: 64 * 4], "big")
    pts[64 * 4: 64 * 5] = pts[64 * 3: 64 * 3 + 32] + (p - y3).to_bytes(32, "big")  # P4 = -P3
    scs = [det_scalar(b"edge", i) for i in range(n)]
    scs[1] = 0
    scs[4] = scs[3]                                        # s*P3 + s*(-P3) cancels
    scs[6] = O.SECP256K1.n + 5                             # unreduced scalar
    sc = b"".join(s.to_bytes(32, "little") for s in scs)
    ok, xy, sec1 = loader.secp_ref_msm(sc, bytes(pts), n)
    out["edge"] = {"n": n, "scalars": sc.hex(), "points": bytes(pts).hex(), "sec1": sec1.hex(), "xy": xy.hex()}
    kat = C.create_string_buffer(32)
    cnt = lib.ref_secp_kat(kat, None)
    out["kat"] = {"source": "tests.c:4715-4757 test_ecmult_constants, expected32 at tests.c:4732-4737",
                  "count": cnt, "sha256": kat.raw.hex()}
    assert kat.raw.hex() == "e4711b4d141e6848b7af472b4cd204143a7587601af96360d0cb1faa859ab7b4"
    return out


def secp_config4_vector():
    """BASELINE config 4 (2^18 terms, the inputs of bench.py's secp256k1 block), computed with the big-int oracle, which
    reproduces the reference's ecmult_multi_var outputs of secp256k1_ref.json.  Takes about a minute."""
    c = O.SECP256K1
    n = 1 << 18
    q = int.from_bytes(hashlib.sha256(b"porla-seed").digest(), "big")
    Q = O.mul(c, q, (c.gx, c.gy))
    pts, cur = [], (c.gx, c.gy)
    for _ in range(n):
        pts.append(cur)
        cur = O.add(c, cur, Q)
    sc = [int.from_bytes(hashlib.sha256(b"cfg4" + i.to_bytes(4, "little")).digest(), "little") for i in range(n)]
    r = O.msm(c, sc, pts, window=12)
    be = lambda v: v.to_bytes(32, "big")
    return {"source": "oracle/curves_py.py msm (big-int oracle; pinned to the reference's ecmult_multi_var by secp256k1_ref.json)",
            "inputs": "points: P0 = G, P(i+1) = P(i) + q*G with q = sha256('porla-seed'); scalars: sha256('cfg4' || LE32(i)) "
                      "as 32 little-endian bytes, NOT reduced",
            "n": n, "chain_sha256": hashlib.sha256(b"".join(be(x) + be(y) for x, y in pts)).hexdigest(),
            "xy": (be(r[0]) + be(r[1])).hex(), "sec1": O.secp_sec1_compressed(r).hex()}


def bn254_vectors():
    c = O.BN254
    G = (1, 2)
    out = {"source": "oracle/curves_py.py (independent big-int restatement; PARITY UNPINNED vs gnark-crypto v0.6.0) "
                     "+ public constants checked in SURVEY.md 8(c)",
           "two_g": O.bn254_marshal(O.mul(c, 2, G)).hex(),
           "tau_g": O.bn254_marshal(O.mul(c, 0xffeeddccbbaa99887766554433221100, G)).hex(),
           "inputs": "points: hash_point(BN254, i) (SURVEY 8(d) recipe); scalars: sha256('porla-sc'||LE64(i)) as a "
                     "256-bit big-endian integer (NOT reduced: fr.SetBytes reduces)",
           "cases": []}
    nmax = 766
    pts = [O.hash_point(c, i) for i in range(nmax)]
    out["points_sha256"] = hashlib.sha256(b"".join(O.bn254_marshal(P) for P in pts)).hexdigest()
    for n in (1, 2, 128, 766):
        sc = [det_scalar(b"porla-sc", i) for i in range(n)]
        out["cases"].append({"n": n, "kind": "uniform256", "marshal": O.bn254_marshal(O.msm(c, sc, pts[:n])).hex()})
    for n in (128, 766):  # Porla audit shape: 31-bit coefficients (Client.hpp:700)
        sc = [det_scalar(b"porla-31", i) & 0x7FFFFFFF for i in range(n)]
        out["cases"].append({"n": n, "kind": "audit31", "marshal": O.bn254_marshal(O.msm(c, sc, pts[:n])).hex()})
    # KZG over the Porla keys (config.hpp:38-39): SRS prefix, a commitment and an opening
    tau = 0xffeeddccbbaa99887766554433221100
    srs = O.kzg_srs_g1(tau, 16)
    f = [det_scalar(b"porla-poly", i) for i in range(16)]
    fr = [x % c.n for x in f]
    y, h = O.kzg_open(fr, 0x1234567)
    out["kzg"] = {"n": 16, "tau": hex(tau), "z": 0x1234567,
                  "srs_compressed": b"".join(O.bn254_compress(P) for P in srs).hex(),
                  "commit": O.bn254_marshal(O.kzg_commit(fr, srs)).hex(),
                  "claim": y.to_bytes(32, "big").hex(),
                  "H": O.bn254_marshal(O.kzg_commit(h, srs[:15])).hex()}
    return out


MAKERS = {"secp256k1_ref": secp_vectors, "bn254": bn254_vectors, "secp256k1_config4": secp_config4_vector}

if __name__ == "__main__":
    for name in sys.argv[1:] or MAKERS:        # e.g. `make_golden.py secp256k1_config4` needs no reference build
        with open(os.path.join(HERE, name + ".json"), "w") as f:
            json.dump(MAKERS[name](), f, indent=1)
    print("wrote golden vectors")
