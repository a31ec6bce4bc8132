"""The data side of an IPA-mode server on the B200: align_MAC and the audit's aggregation over resident secp256k1
generators, and the multi-exponentiation of Jacobian MACs as stored.  Generators are g_i = k_i G, so every commitment
has the closed form [sum x_i k_i mod n] G.  The align_MAC arithmetic is checked against its restatement
(mod = A % PRIME_MODULUS, c = (mod - A) % n) and, independently of it, against the protocol identity
sum (A_i mod n) g_i + align = sum (A_i mod PRIME_MODULUS) g_i."""
import ctypes as C
import random
import threading

import pytest

import porla_b200 as pb
from oracle import curves_py as O
from tests.common import le
from tests.test_secp_butterfly import SE, G, from_gej, to_gej

pytestmark = pytest.mark.gpu

PRIME = 207 * 2**248 + 1            # PRIME_MODULUS, utils.h:40
LCM = PRIME * SE.n                  # LCM_IPA, utils.h:32
EDGES = [0, PRIME, PRIME - 1, LCM - 1, SE.n, 7 * PRIME + 3]


def commit(ks, xs):
    """sum x_i g_i for g_i = k_i G, in closed form; None for infinity."""
    s = sum(x * k for x, k in zip(xs, ks)) % SE.n
    return O.mul(SE, s, G) if s else None


_GENS = {}


def generators(count, with_u):
    """(discrete logs, resident table): `count` generators, followed by u when with_u (the prover's table)."""
    key = (count, with_u)
    if key not in _GENS:
        rnd = random.Random(count * 2 + with_u)
        ks = [rnd.randrange(1, SE.n) for _ in range(count + with_u)]
        _GENS[key] = (ks, pb.SecpGenerators([O.mul(SE, k, G) for k in ks]))
    return _GENS[key]


def align_blocks(batch, n_chunks, seed):
    rnd = random.Random(seed)
    vals = [[rnd.randrange(LCM) for _ in range(n_chunks)] for _ in range(batch)]
    vals[0][:len(EDGES)] = EDGES
    if batch > 1:
        vals[-1] = [rnd.randrange(PRIME) for _ in range(n_chunks)]      # already reduced: alignment is infinity
    return vals


def to_data(vals):
    return bytearray(b"".join(v.to_bytes(64, "little") for row in vals for v in row))


@pytest.mark.parametrize("batch", [1, 8, 9, 1024])
@pytest.mark.parametrize("table", ["gens128", "gens_u129"])
def test_align_mac_batch_against_restatement_and_protocol_identity(table, batch):
    with_u = table == "gens_u129"
    n_chunks = 100 if with_u else 128
    ks, tab = generators(128, with_u)
    vals = align_blocks(batch, n_chunks, 31 * batch + n_chunks)
    data = to_data(vals)
    ok, out = tab.align_mac_batch(data, batch, n_chunks)
    assert ok == 1
    got = from_gej(out[:batch])
    want_data = b"".join((v % PRIME).to_bytes(32, "little") + bytes(32) for row in vals for v in row)
    assert bytes(data) == want_data
    rnd = random.Random(batch)
    checked = range(batch) if batch <= 9 else sorted({0, batch - 1} | set(rnd.sample(range(batch), 30)))
    for b in checked:
        c = [((v % PRIME) - v) % SE.n for v in vals[b]]
        assert got[b] == commit(ks, c), b
    if batch > 1:
        assert got[-1] is None
    # the identity the server relies on, with the library's own commitments on both sides
    for b in list(checked)[:3]:
        lhs_ok, lhs = tab.multi(0, [v % SE.n for v in vals[b]])
        rhs_ok, rhs = tab.multi(0, [v % PRIME for v in vals[b]])
        assert lhs_ok == rhs_ok == 1
        assert O.add(SE, lhs, got[b]) == rhs, b


def test_align_mac_batch_shapes_and_empty_call():
    ks, tab = generators(128, False)
    bn = pb.Table.multiples_of_generator(pb.CURVE_BN254, b"".join(le(k) for k in ks[:128]), 128)
    lib = pb.load()
    vals = align_blocks(2, 128, 5)
    for handle, n_chunks in ((tab.handle, 0), (tab.handle, 129), (bn.handle, 128), (None, 128)):
        data = to_data(vals)
        out = (pb.lib.SecpGej * 2)()
        C.memset(out, 0x5A, C.sizeof(out))
        before = bytes(out)
        assert lib.porla_secp256k1_align_mac_batch(handle, n_chunks, pb.lib._as_void_p(data), 2, out) == 0
        assert bytes(data) == bytes(to_data(vals)) and bytes(out) == before, n_chunks
    out = (pb.lib.SecpGej * 1)()
    C.memset(out, 0x5A, C.sizeof(out))
    before = bytes(out)
    assert lib.porla_secp256k1_align_mac_batch(tab.handle, 128, None, 0, out) == 1
    assert bytes(out) == before
    bn.destroy()


@pytest.mark.parametrize("n", [0, 1, 128, 766])
def test_audit_aggregate_against_restatement_homomorphism_and_prover(n):
    from oracle import ipa_py
    n_chunks = 128
    ks, tab = generators(128, True)
    rnd = random.Random(766 + n)
    coefs = [rnd.randrange(1 << 31) for _ in range(n)]
    blocks = [[rnd.randrange(LCM) for _ in range(n_chunks)] for _ in range(n)]
    if n:
        coefs[0] = (1 << 31) - 1
        blocks[0][:len(EDGES)] = EDGES
    if n > 2:
        coefs[1] = 0
    for row in blocks:
        row[7] = LCM - 1                                           # the widest possible sum in chunk 7
    ok, b_out, al = tab.audit_aggregate(b"".join(c.to_bytes(4, "little") for c in coefs),
                                        b"".join(v.to_bytes(64, "little") for row in blocks for v in row), n, n_chunks)
    assert ok == 1
    align = from_gej([al])[0]
    B = [sum(c * row[j] for c, row in zip(coefs, blocks)) for j in range(n_chunks)]
    got_b = [int.from_bytes(b_out[32 * j:32 * j + 32], "little") for j in range(n_chunks)]
    assert got_b == [b % PRIME for b in B]
    assert align == commit(ks, [((b % PRIME) - b) % SE.n for b in B])
    # sum_j coef_j commit(block_j) + align = commit(b_out), the commitments by the library
    lin_ok, lin = tab.multi(0, [b % SE.n for b in B])
    out_ok, com_b = tab.multi(0, got_b)
    assert lin_ok == out_ok == 1 and O.add(SE, lin, align) == com_b
    if n == 128:                                                   # b_out is the prover's `a` as it stands
        gens, u = [O.mul(SE, k, G) for k in ks[:n_chunks]], O.mul(SE, ks[n_chunks], G)
        bv = [rnd.randrange(SE.n) for _ in range(n_chunks)]
        assert tab.inner_product_prove(got_b, bv) == ipa_py.inner_product_prove(gens, u, got_b, bv)


def test_audit_aggregate_shapes():
    ks, tab = generators(128, True)
    lib = pb.load()
    coefs, blocks = bytearray(8), bytearray(2 * 128 * 64)
    for handle, n_chunks, n in ((tab.handle, 0, 2), (tab.handle, 130, 2), (tab.handle, 128, 1 << 24), (None, 128, 2)):
        b_out = bytearray(b"\x5a" * 32 * 130)
        al = pb.lib.SecpGej()
        C.memset(C.byref(al), 0x5A, C.sizeof(al))
        assert lib.porla_secp256k1_audit_aggregate(handle, n_chunks, pb.lib._as_void_p(coefs), pb.lib._as_void_p(blocks), n,
                                                   pb.lib._as_void_p(b_out), C.byref(al)) == 0
        assert b_out == bytearray(b"\x5a" * 32 * 130) and bytes(al) == b"\x5a" * C.sizeof(al), (n_chunks, n)


# ---------------------------------------------------------------------------- MACs as stored
def gej_case(n, nbatch, seed):
    """(discrete logs, scalars, affine points) for nbatch MSMs of n terms with infinities, zero scalars, scalars >= n and,
    in the second MSM, a combination that cancels to infinity.  Points come from a device table of k_i G."""
    rnd = random.Random(seed)
    total = n * nbatch
    ks = [rnd.randrange(1, SE.n) for _ in range(total)]
    sc = [rnd.randrange(1 << 256) for _ in range(total)]
    for i in range(0, total, 97):
        ks[i] = 0                                                  # infinity
    for i in range(1, total, 89):
        sc[i] = 0
    for i in range(2, total, 83):
        sc[i] = SE.n + rnd.randrange(1 << 32)                      # >= n, taken mod n
    if nbatch > 1:                                                 # MSM 1 cancels: sum s_i k_i = 0 mod n
        lo, hi = n, 2 * n
        if ks[hi - 1] == 0:
            ks[hi - 1] = 3
        rest = sum(s * k for s, k in zip(sc[lo:hi - 1], ks[lo:hi - 1]))
        v = -rest * pow(ks[hi - 1], -1, SE.n) % SE.n
        sc[hi - 1] = v + SE.n if v + SE.n < 1 << 256 else v             # >= n as well where a 256-bit scalar allows it
    tab = pb.Table.multiples_of_generator(pb.CURVE_SECP256K1, b"".join(le(k) for k in ks), total)
    raw = tab.export(pb.POINT_LE64)
    tab.destroy()
    pts = []
    for i in range(total):
        rec = raw[64 * i:64 * i + 64]
        pts.append(None if rec == bytes(64) else (int.from_bytes(rec[:32], "little"), int.from_bytes(rec[32:], "little")))
    return ks, sc, pts


def drop_in(scalars, points):
    """porla_secp256k1_ecmult_multi_var over the same points as secp256k1_ge, its raw 128-byte result."""
    def cb(sc_p, pt_p, idx, _data):
        s = scalars[idx]
        for i in range(4):
            sc_p.contents.d[i] = (s >> (64 * i)) & 0xFFFFFFFFFFFFFFFF
        P = points[idx]
        C.memset(pt_p, 0, C.sizeof(pb.lib.SecpGe))
        if P is None:
            pt_p.contents.infinity = 1
        else:
            pt_p.contents.x, pt_p.contents.y = pb.lib._int_to_fe(P[0]), pb.lib._int_to_fe(P[1])
        return 1

    r = pb.lib.SecpGej()
    assert pb.load().porla_secp256k1_ecmult_multi_var(None, None, C.byref(r), None, pb.lib.SECP_CB(cb), None, len(scalars)) == 1
    return bytes(r)


@pytest.mark.parametrize("nbatch", [1, 2])
@pytest.mark.parametrize("n", [1, 128, 766, (1 << 17) + 3])
def test_gej_multi_exponentiation_against_closed_form_and_drop_in(n, nbatch):
    ks, sc, pts = gej_case(n, nbatch, 17 * n + nbatch)
    gejs = to_gej(pts, random.Random(n))
    before = bytes(gejs)
    ok, r = pb.secp256k1_ecmult_multi_gej(gejs, sc, n, nbatch)
    assert ok == 1 and bytes(gejs) == before
    got = from_gej(r[:nbatch])
    for b in range(nbatch):
        part = slice(b * n, (b + 1) * n)
        assert got[b] == commit(ks[part], sc[part]), b
        assert bytes(r[b]) == drop_in(sc[part], pts[part]), b
    if nbatch > 1:
        assert got[1] is None


def test_concurrent_aligns_and_gej_calls_equal_their_serial_values():
    """Porla's pool threads (Server.hpp:1077-1078) issue align_MAC per block; the audit's multi-exponentiations run
    alongside.  Eight threads, each with its own blocks and MACs, several rounds: every result equals the serial one."""
    ks, tab = generators(128, False)
    T, rounds = 8, 4
    blocks = [align_blocks(1, 128, 900 + t) for t in range(T)]
    cases = [gej_case(128, 1, 700 + t) for t in range(T)]
    gejs = [to_gej(pts, random.Random(t)) for t, (_, _, pts) in enumerate(cases)]
    want_align, want_data, want_gej = [], [], []
    for t in range(T):
        data = to_data(blocks[t])
        ok, out = tab.align_mac_batch(data, 1, 128)
        assert ok == 1
        want_align.append(bytes(out[0]))
        want_data.append(bytes(data))
        ok, r = pb.secp256k1_ecmult_multi_gej(gejs[t], cases[t][1], 128, 1)
        assert ok == 1
        want_gej.append(bytes(r[0]))
    errors = []

    def worker(t):
        for _ in range(rounds):
            data = to_data(blocks[t])
            ok, out = tab.align_mac_batch(data, 1, 128)
            if ok != 1 or bytes(out[0]) != want_align[t] or bytes(data) != want_data[t]:
                errors.append(("align", t))
            ok, r = pb.secp256k1_ecmult_multi_gej(gejs[t], cases[t][1], 128, 1)
            if ok != 1 or bytes(r[0]) != want_gej[t]:
                errors.append(("gej", t))

    th = [threading.Thread(target=worker, args=(t,)) for t in range(T)]
    [x.start() for x in th]
    [x.join() for x in th]
    assert not errors, errors[:6]
    assert want_align[0] != want_align[1] and want_gej[0] != want_gej[1]
