"""Every staged host-buffer entry point gives the same bytes whether a call leases a staging slot of its own or takes the
shared staging area under the global mutex (PORLA_SERIAL_CALLS=1, read per call), on shapes on both sides of the slot
limits: 4096 / 4097 terms and 4 / 5 MSMs per call.  Results also equal closed forms: every point has a known discrete
logarithm (chains P_i = (a + i q) G, the SRS [tau^i] G1), so an MSM is one scalar multiplication of the generator."""
import ctypes as C
import random

import pytest

import porla_b200 as pb
from oracle import curves_py as O
from tests.test_secp_butterfly import to_gej

pytestmark = pytest.mark.gpu

BN, SE = O.BN254, O.SECP256K1
TAU = bytes.fromhex("ffeeddccbbaa99887766554433221100")
ALPHA = bytes.fromhex("00112233445566778899aabbccddeeff")
TAU_I, ALPHA_I = int.from_bytes(TAU, "big") % BN.n, int.from_bytes(ALPHA, "big") % BN.n
PRIME = 207 * 2**248 + 1            # PRIME_MODULUS, utils.h:40
FIRST = 3                           # table sub-range calls start inside the table
# (n, nbatch): a slot at the term limit, the shared area past it, a slot at the batch limit, the shared area past it
SHAPES = [(4096, 1), (4097, 1), (1024, 4), (16, 5)]


def enc(P):
    return bytes(64) if P is None else P[0].to_bytes(32, "big") + P[1].to_bytes(32, "big")


def gen(c):
    return (c.gx, c.gy)


CHAIN_LEN = FIRST + 4097
_CHAINS = {}


def chain(c, count):
    """(logs, points) with points[i] = logs[i] G, the same prefix for every count: additions only."""
    if c.name not in _CHAINS:
        a, q = 0x5EED, 0xC0FFEE1234567
        P, Q, pts = O.mul(c, a, gen(c)), O.mul(c, q, gen(c)), []
        for _ in range(CHAIN_LEN):
            pts.append(P)
            P = O.add(c, P, Q)
        _CHAINS[c.name] = ([(a + i * q) % c.n for i in range(CHAIN_LEN)], pts)
    logs, pts = _CHAINS[c.name]
    return logs[:count], pts[:count]


def commit(c, logs, scalars):
    return O.mul(c, sum(s * k for s, k in zip(scalars, logs)) % c.n, gen(c))


def ints(rnd, count, bound=1 << 256):
    return [rnd.randrange(bound) for _ in range(count)]


def be32(vals):
    return b"".join(v.to_bytes(32, "big") for v in vals)


def le32(vals):
    return b"".join(v.to_bytes(32, "little") for v in vals)


def buf(b):
    return pb.lib._as_void_p(b)


_KZG = {}


def kzg(n):
    """A Kzg state with an n-point SRS; re-initialised only when n changes."""
    if _KZG.get("n") != n:
        _KZG["k"] = pb.Kzg(TAU, ALPHA)
        _KZG["k"].init_srs(n)
        _KZG["n"] = n
    return _KZG["k"]


def poly_at(coeffs, x):
    return sum(f * pow(x, i, BN.n) for i, f in enumerate(coeffs)) % BN.n


_TABLES = {}


def table(c, count):
    """A resident table of the first `count` chain points (secp256k1: expanded like Porla's generators)."""
    if (c.name, count) not in _TABLES:
        pts = chain(c, count)[1]
        _TABLES[c.name, count] = (pb.SecpGenerators(pts) if c is SE else
                                  pb.Table.from_host(pb.CURVE_BN254, b"".join(enc(P) for P in pts)))
    return _TABLES[c.name, count]


# Each case returns (call, want): call() runs the entry point and returns its output bytes; want is what they must be.
def msm_host(curve_id, c, fmt, enc_out):
    def case(n, nbatch, rnd):
        logs, pts = chain(c, n * nbatch)
        sc = ints(rnd, n * nbatch)
        scalars = (be32 if fmt == pb.SCALAR_BE32 else le32)(sc)
        points = b"".join(enc_out(P) for P in pts)
        want = b"".join(enc_out(commit(c, logs[b * n:(b + 1) * n], sc[b * n:(b + 1) * n])) for b in range(nbatch))
        return lambda: pb.msm_host(curve_id, scalars, points, n, nbatch, scalar_fmt=fmt,
                                   point_fmt=pb.POINT_BE64 if enc_out is enc else pb.POINT_LE64), want
    return case


def le_point(P):
    return bytes(64) if P is None else P[0].to_bytes(32, "little") + P[1].to_bytes(32, "little")


def digest_from_srs(n, nbatch, rnd):
    k = kzg(n)
    f = ints(rnd, n * nbatch)
    want = b"".join(enc(O.mul(BN, poly_at(f[b * n:(b + 1) * n], TAU_I), gen(BN))) for b in range(nbatch))
    if nbatch == 1:
        return lambda: k.compute_digest_from_srs(be32(f)), want
    return lambda: k.compute_digest_from_srs_batch(be32(f), nbatch), want


def create_proof(n, nbatch, rnd):
    """Two commitments in one call: f and its quotient by (x - z)."""
    k = kzg(n)
    f, z = ints(rnd, n, BN.n), rnd.randrange(1 << 64)
    y = poly_at(f, z)
    h = (poly_at(f, TAU_I) - y) * pow(TAU_I - z, -1, BN.n) % BN.n
    want = enc(O.mul(BN, poly_at(f, TAU_I), gen(BN))) + enc(O.mul(BN, h, gen(BN))) + be32([z, y])
    return lambda: b"".join(k.create_proof(z, be32(f))), want


def table_host_scalars(n, nbatch, rnd):
    logs = chain(BN, FIRST + n)[0]
    tab = table(BN, CHAIN_LEN)
    sc = ints(rnd, n * nbatch)
    want = b"".join(enc(commit(BN, logs[FIRST:], sc[b * n:(b + 1) * n])) for b in range(nbatch))
    scalars = le32(sc)

    def call():
        out = bytearray(64 * nbatch)
        pb.load().porla_msm_table_host_scalars_batch(C.c_void_p(tab.handle), FIRST, buf(scalars), n, nbatch, pb.SCALAR_LE32,
                                                     pb.POINT_BE64, buf(out))
        return bytes(out)
    return call, want


def digest_batch(n, nbatch, rnd):
    k = kzg(n)
    f = ints(rnd, n * nbatch)
    want = b"".join(enc(O.mul(BN, ALPHA_I * poly_at(f[b * n:(b + 1) * n], TAU_I), gen(BN))) for b in range(nbatch))
    return lambda: k.compute_digest_batch(be32(f), nbatch), want


def digest_complement_batch(n, nbatch, rnd):
    k = kzg(n)
    s = ints(rnd, nbatch)
    want = b"".join(k.compute_digest_complement(be32([v])) for v in s)   # the per-call host symbol
    return lambda: k.compute_digest_complement_batch(be32(s), nbatch), want


def align_values(rnd, count, modulus):
    vals = ints(rnd, count, PRIME * modulus)
    vals[:3] = [0, PRIME, PRIME * modulus - 1]
    return vals


def bn254_align_mac(n, nbatch, rnd):
    k = kzg(n)
    vals = align_values(rnd, n * nbatch, BN.n)
    srs_logs = [pow(TAU_I, i, BN.n) for i in range(n)]
    want = b"".join(enc(commit(BN, srs_logs, [(v % PRIME - v) % BN.n for v in vals[b * n:(b + 1) * n]]))
                    for b in range(nbatch)) + b"".join((v % PRIME).to_bytes(64, "little") for v in vals)

    def call():
        data = bytearray(b"".join(v.to_bytes(64, "little") for v in vals))
        return k.align_mac_batch(data, nbatch) + bytes(data)
    return call, want


def audit_inputs(rnd, chunks, blocks, modulus):
    coefs = ints(rnd, blocks, 1 << 31)
    rows = [align_values(rnd, chunks, modulus) for _ in range(blocks)]
    B = [sum(cf * row[j] for cf, row in zip(coefs, rows)) for j in range(chunks)]
    return (b"".join(cf.to_bytes(4, "little") for cf in coefs), b"".join(v.to_bytes(64, "little") for row in rows for v in row),
            B)


def bn254_audit(n, nbatch, rnd):
    """n chunks (the SRS length), nbatch blocks: the call leases by n * nbatch terms."""
    k = kzg(n)
    coefs, blocks, B = audit_inputs(rnd, n, nbatch, BN.n)
    srs_logs = [pow(TAU_I, i, BN.n) for i in range(n)]
    want = be32([b % PRIME for b in B]) + enc(commit(BN, srs_logs, [(b % PRIME - b) % BN.n for b in B]))
    return lambda: b"".join(k.audit_aggregate(coefs, blocks, nbatch)), want


def gej_bytes(ok, arr):
    assert ok == 1
    return bytes(arr)


def secp_want(points):
    """The bytes of a SecpGej array holding `points` as the entries write them (z = 1, normalised limbs)."""
    arr = (pb.lib.SecpGej * len(points))()
    for g, P in zip(arr, points):
        if P is None:
            g.infinity = 1
        else:
            g.x, g.y, g.z, g.infinity = pb.lib._int_to_fe(P[0]), pb.lib._int_to_fe(P[1]), pb.lib._int_to_fe(1), 0
    return bytes(arr)


def secp_align_mac(n, nbatch, rnd):
    logs = chain(SE, n)[0]
    tab = table(SE, CHAIN_LEN)
    vals = align_values(rnd, n * nbatch, SE.n)
    want = secp_want([commit(SE, logs, [(v % PRIME - v) % SE.n for v in vals[b * n:(b + 1) * n]]) for b in range(nbatch)])

    def call():
        data = bytearray(b"".join(v.to_bytes(64, "little") for v in vals))
        out = gej_bytes(*tab.align_mac_batch(data, nbatch, n))
        assert data == b"".join((v % PRIME).to_bytes(64, "little") for v in vals)
        return out
    return call, want


def secp_audit(n, nbatch, rnd):
    logs = chain(SE, n)[0]
    tab = table(SE, CHAIN_LEN)
    coefs, blocks, B = audit_inputs(rnd, n, nbatch, SE.n)
    want = le32([b % PRIME for b in B]) + secp_want([commit(SE, logs, [(b % PRIME - b) % SE.n for b in B])])

    def call():
        ok, b_out, al = tab.audit_aggregate(coefs, blocks, nbatch, n)
        return b_out + gej_bytes(ok, al)
    return call, want


def secp_multi_gej(n, nbatch, rnd):
    logs, pts = chain(SE, n * nbatch)
    gejs = to_gej(pts, rnd)
    sc = ints(rnd, n * nbatch)
    want = secp_want([commit(SE, logs[b * n:(b + 1) * n], sc[b * n:(b + 1) * n]) for b in range(nbatch)])
    return lambda: gej_bytes(*pb.lib.secp256k1_ecmult_multi_gej(gejs, sc, n, nbatch)), want


def secp_const_batch(n, nbatch, rnd):
    """nbatch products of one base: the call leases by its scalar count."""
    (log,), base = chain(SE, 1)[0], table(SE, 1)
    s = ints(rnd, nbatch)
    want = secp_want([O.mul(SE, v * log, gen(SE)) for v in s])

    def call():
        r = (pb.lib.SecpGej * nbatch)()
        ok = pb.load().porla_secp256k1_ecmult_const_batch(C.c_void_p(base.handle), pb.lib._scalar_array(s), nbatch, r)
        return gej_bytes(ok, r)
    return call, want


def secp_table_batch(n, nbatch, rnd):
    logs = chain(SE, CHAIN_LEN)[0]
    tab = table(SE, CHAIN_LEN)
    sc = ints(rnd, n * nbatch)
    want = secp_want([commit(SE, logs[FIRST:FIRST + n], sc[b * n:(b + 1) * n]) for b in range(nbatch)])

    def call():
        r = (pb.lib.SecpGej * nbatch)()
        ok = pb.load().porla_secp256k1_ecmult_multi_table_batch(C.c_void_p(tab.handle), FIRST, pb.lib._scalar_array(sc), n,
                                                                nbatch, r)
        return gej_bytes(ok, r)
    return call, want


ENTRIES = {
    "bn254_msm_host": msm_host(pb.CURVE_BN254, BN, pb.SCALAR_BE32, enc),
    "secp256k1_msm_host": msm_host(pb.CURVE_SECP256K1, SE, pb.SCALAR_LE32, le_point),
    "compute_digest_from_srs": digest_from_srs,
    "create_proof": create_proof,
    "msm_table_host_scalars_batch": table_host_scalars,
    "compute_digest_batch": digest_batch,
    "compute_digest_complement_batch": digest_complement_batch,
    "bn254_align_mac_batch": bn254_align_mac,
    "bn254_audit_aggregate": bn254_audit,
    "secp256k1_align_mac_batch": secp_align_mac,
    "secp256k1_audit_aggregate": secp_audit,
    "secp256k1_ecmult_multi_gej": secp_multi_gej,
    "secp256k1_ecmult_const_batch": secp_const_batch,
    "secp256k1_ecmult_multi_table_batch": secp_table_batch,
}


@pytest.mark.parametrize("n,nbatch", SHAPES)
@pytest.mark.parametrize("entry", list(ENTRIES))
def test_slot_and_shared_staging_give_the_same_bytes(entry, n, nbatch, monkeypatch):
    pb.load().porla_device_init()
    monkeypatch.delenv("PORLA_SERIAL_CALLS", raising=False)
    call, want = ENTRIES[entry](n, nbatch, random.Random(f"{entry}/{n}/{nbatch}"))
    slot = call()
    monkeypatch.setenv("PORLA_SERIAL_CALLS", "1")
    shared = call()
    assert slot == shared
    assert slot == want
