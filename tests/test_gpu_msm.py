"""Parity of the CUDA path against the oracle, through the C-ABI (libmultiexp.so).

BN254: the oracle is oracle/curves_py.py (independent big-int restatement; gnark-crypto is not
available, so "parity vs restatement").  secp256k1: oracle/curves_py.py here, and the vendored
reference C (oracle/_ref) in tests/test_gpu_secp_ref.py.
"""
import ctypes as C
import random

import pytest

import porla_b200 as pb
from oracle import curves_py as O

pytestmark = pytest.mark.gpu

BN, SE = O.BN254, O.SECP256K1


def be(x):
    return x.to_bytes(32, "big")


def enc_points(pts):
    return b"".join(bytes(64) if P is None else be(P[0]) + be(P[1]) for P in pts)


def rand_points(c, n, seed):
    rnd = random.Random(seed)
    G = (c.gx, c.gy)
    base = [O.hash_point(c, i) for i in range(min(n, 24))]
    out = []
    for i in range(n):
        if i < len(base):
            out.append(base[i])
        else:  # cheap: sums of earlier points stay on the curve
            out.append(O.add(c, out[rnd.randrange(i)], out[rnd.randrange(i)]))
    return out


@pytest.mark.parametrize("curve,c", [(pb.CURVE_BN254, BN), (pb.CURVE_SECP256K1, SE)])
def test_field_mul_matches_bigint(curve, c):
    rnd = random.Random(1)
    n = 4096
    a = [rnd.randrange(c.p) for _ in range(n)]
    b = [rnd.randrange(c.p) for _ in range(n)]
    a[0], b[0] = c.p - 1, c.p - 1
    a[1], b[1] = 0, 5
    a[2], b[2] = 1, c.p - 1
    # values that drive the special-form folds / the last Montgomery subtraction to their corners
    edge = [0, 1, 2, c.p - 1, c.p - 2, (1 << 255) % c.p, (1 << 32) - 1, ((1 << 256) - 1) % c.p, c.p >> 1,
            (1 << 224) - 1, c.p - (1 << 32), (c.p + 1) // 2]
    for i, (x, y) in enumerate((x, y) for x in edge for y in edge):
        a[3 + i], b[3 + i] = x, y
    le = lambda v: v.to_bytes(32, "little")
    ab, bb, ob = bytearray(b"".join(map(le, a))), bytearray(b"".join(map(le, b))), bytearray(32 * n)
    pb.load().porla_debug_field_mul(curve, (C.c_ubyte * len(ab)).from_buffer(ab), (C.c_ubyte * len(bb)).from_buffer(bb), n,
                                    (C.c_ubyte * len(ob)).from_buffer(ob))
    rinv = pow(1 << 256, -1, c.p) if c is BN else 1
    for i in range(n):
        got = int.from_bytes(ob[32 * i:32 * i + 32], "little")
        assert got == a[i] * b[i] * rinv % c.p, i


@pytest.mark.parametrize("curve,c", [(pb.CURVE_BN254, BN), (pb.CURVE_SECP256K1, SE)])
@pytest.mark.parametrize("op", [1, 2])
def test_field_square_and_product_sum_match_bigint(curve, c, op):
    """The dedicated squaring (36 products) and the fused product-sum a*b + b*(a+b) (one reduction)
    that the bucket update uses, on edge values and random residues."""
    rnd = random.Random(10 + op)
    n = 4096
    a = [rnd.randrange(c.p) for _ in range(n)]
    b = [rnd.randrange(c.p) for _ in range(n)]
    edge = [0, 1, 2, c.p - 1, c.p - 2, (1 << 255) % c.p, (1 << 32) - 1, ((1 << 256) - 1) % c.p, c.p >> 1]
    for i, (x, y) in enumerate((x, y) for x in edge for y in edge):
        a[i], b[i] = x, y
    le = lambda v: v.to_bytes(32, "little")
    ab, bb, ob = bytearray(b"".join(map(le, a))), bytearray(b"".join(map(le, b))), bytearray(32 * n)
    pb.load().porla_debug_field_op(curve, op, (C.c_ubyte * len(ab)).from_buffer(ab), (C.c_ubyte * len(bb)).from_buffer(bb), n,
                                   (C.c_ubyte * len(ob)).from_buffer(ob))
    rinv = pow(1 << 256, -1, c.p) if c is BN else 1
    for i in range(n):
        got = int.from_bytes(ob[32 * i:32 * i + 32], "little")
        want = a[i] * a[i] if op == 1 else a[i] * b[i] + b[i] * ((a[i] + b[i]) % c.p)
        assert got == want * rinv % c.p, (i, op)


@pytest.mark.parametrize("n", [1, 2, 3, 17, 128, 766, 1500])
def test_compute_multi_exp_matches_oracle(n):
    rnd = random.Random(n)
    pts = rand_points(BN, n, n)
    sc = [rnd.randrange(1 << 256) for _ in range(n)]          # >= r values are reduced (fr.SetBytes)
    got = pb.bn254_multi_exp(enc_points(pts), b"".join(map(be, sc)), n)
    assert got == O.bn254_marshal(O.msm(BN, sc, pts))


def test_compute_multi_exp_zero_length():
    assert pb.bn254_multi_exp(b"", b"", 0) == bytes(64)


def test_porla_audit_shape_31bit_scalars_with_infinities():
    # Server.hpp:900-901: 31-bit coefficients, many alignment MACs still infinity
    n = 766
    rnd = random.Random(7)
    pts = rand_points(BN, n, 3)
    for i in range(0, n, 5):
        pts[i] = None
    sc = [rnd.randrange(1 << 31) for _ in range(n)]
    scb = b"".join(pb.bn254_scalar_set_int(s) for s in sc)
    got = pb.bn254_multi_exp(enc_points(pts), scb, n)
    assert got == O.bn254_marshal(O.msm(BN, sc, pts))


def test_edge_cases_cancel_duplicate_zero():
    rnd = random.Random(11)
    P, Q = O.hash_point(BN, 100), O.hash_point(BN, 101)
    cases = [
        ([5, 5], [P, O.neg(BN, P)]),                 # cancels to infinity
        ([3, 4, 9], [P, P, P]),                      # same point in several buckets
        ([7, 7, 7, 7], [P, P, Q, Q]),                # P + P inside one bucket -> doubling branch
        ([0, 0, 0], [P, Q, P]),                      # all-zero scalars
        ([BN.n, BN.n + 1], [P, Q]),                  # reduction: r -> 0, r+1 -> 1
        ([BN.n - 1, 1], [P, P]),                     # (r-1)P + P = infinity
        ([1 << 255, (1 << 256) - 1], [P, Q]),
        ([12345], [None]),
    ]
    for sc, pts in cases:
        got = pb.bn254_multi_exp(enc_points(pts), b"".join(map(be, sc)), len(sc))
        assert got == O.bn254_marshal(O.msm_naive(BN, sc, pts)), (sc,)
    # constant scalar, many points (one giant bucket per window)
    n = 300
    pts = rand_points(BN, n, 5)
    k = rnd.randrange(BN.n)
    got = pb.bn254_multi_exp(enc_points(pts), be(k) * n, n)
    assert got == O.bn254_marshal(O.msm(BN, [k] * n, pts))


def test_batch_multi_exp():
    batch, n = 5, 40
    rnd = random.Random(3)
    pts = rand_points(BN, batch * n, 9)
    sc = [rnd.randrange(BN.n) for _ in range(batch * n)]
    got = pb.bn254_multi_exp_batch(enc_points(pts), b"".join(map(be, sc)), n, batch)
    for m in range(batch):
        exp = O.bn254_marshal(O.msm(BN, sc[m * n:(m + 1) * n], pts[m * n:(m + 1) * n]))
        assert got[64 * m:64 * m + 64] == exp, m


@pytest.mark.parametrize("window", [0, 4, 9, 13, 16])
def test_window_sizes_agree(window, monkeypatch):
    n = 600
    rnd = random.Random(2)
    pts = rand_points(BN, n, 21)
    sc = [rnd.randrange(BN.n) for _ in range(n)]
    if window:
        monkeypatch.setenv("PORLA_WINDOW_BITS", str(window))
    got = pb.bn254_multi_exp(enc_points(pts), b"".join(map(be, sc)), n)
    assert got == O.bn254_marshal(O.msm(BN, sc, pts))


@pytest.mark.parametrize("switch", ["PORLA_REDUCE_V1=1", "PORLA_SORT_V2=0", "PORLA_SORT_V2=1"])
@pytest.mark.parametrize("n,window", [(600, 9), (5000, 0), (70001, 0), ((1 << 19) + 5, 0)])
def test_opt_in_kernel_variants_agree(switch, n, window, monkeypatch):
    """The variants behind environment switches (profiles/r02*): the round-1 bucket reduction and the sort with / without
    the exact histogram.  Same bytes as the default pipeline; the large
    sizes go through the resident path with points k_i G and the closed form (sum s_i k_i) G."""
    import torch
    rnd = random.Random(n)
    if window:
        monkeypatch.setenv("PORLA_WINDOW_BITS", str(window))
    if n <= 5000:
        pts = rand_points(BN, n, 5)
        sc = [rnd.randrange(1 << 256) for _ in range(n)]
        args = (enc_points(pts), b"".join(map(be, sc)), n)
        want = pb.bn254_multi_exp(*args)
        assert want == O.bn254_marshal(O.msm(BN, sc, pts))
        monkeypatch.setenv(*switch.split("="))
        assert pb.bn254_multi_exp(*args) == want
        return
    g = torch.Generator(device="cuda")
    g.manual_seed(n)
    ks = torch.randint(0, 2**31 - 1, (n, 8), dtype=torch.int32, device="cuda", generator=g)
    ks[:, 1:] = 0
    ss = torch.randint(-2**31, 2**31 - 1, (n, 8), dtype=torch.int32, device="cuda", generator=g)
    tab = pb.Table.multiples_of_generator(pb.CURVE_BN254, ks.data_ptr(), n, pb.SCALAR_LE32, on_device=True)
    kv = ks[:, 0].cpu().numpy().astype("uint32").tolist()
    sv = ss.cpu().numpy().view("uint32")
    total = sum(k * sum(int(v) << (32 * j) for j, v in enumerate(row)) for k, row in zip(kv, sv.tolist())) % BN.n
    want = O.bn254_marshal(O.mul(BN, total, (1, 2)))
    assert tab.msm_resident(ss.data_ptr(), n, scalar_fmt=pb.SCALAR_LE32) == want
    monkeypatch.setenv(*switch.split("="))
    assert tab.msm_resident(ss.data_ptr(), n, scalar_fmt=pb.SCALAR_LE32) == want
    tab.destroy()


def test_multiples_table_and_closed_form():
    # table[i] = k_i G; MSM(s, table) = (sum s_i k_i) G  -- size-independent checksum
    import torch
    n = 1 << 14
    rnd = random.Random(4)
    ks = [rnd.randrange(BN.n) for _ in range(n)]
    ss = [rnd.randrange(BN.n) for _ in range(n)]
    tab = pb.Table.multiples_of_generator(pb.CURVE_BN254, b"".join(k.to_bytes(32, "little") for k in ks), n, pb.SCALAR_LE32)
    ext = tab.export()
    G = (1, 2)
    for i in (0, 1, n // 2, n - 1):
        assert ext[64 * i:64 * i + 64] == O.bn254_marshal(O.mul(BN, ks[i], G))
    d_sc = torch.frombuffer(bytearray(b"".join(map(be, ss))), dtype=torch.uint8).cuda()
    d_out = torch.zeros(64, dtype=torch.uint8, device="cuda")
    tab.msm_device(d_sc.data_ptr(), n, d_out.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    expect = O.mul(BN, sum(s * k for s, k in zip(ss, ks)) % BN.n, G)
    assert bytes(d_out.cpu().numpy()) == O.bn254_marshal(expect)
    tab.destroy()


@pytest.mark.parametrize("n", [1, 5, 96, 700])
def test_secp256k1_msm_host(n):
    rnd = random.Random(n + 1)
    pts = rand_points(SE, n, n + 5)
    sc = [rnd.randrange(1 << 256) for _ in range(n)]
    got = pb.msm_host(pb.CURVE_SECP256K1, b"".join(s.to_bytes(32, "little") for s in sc), enc_points(pts), n,
                      scalar_fmt=pb.SCALAR_LE32, point_fmt=pb.POINT_BE64)
    exp = O.msm(SE, sc, pts)
    assert got == (bytes(64) if exp is None else be(exp[0]) + be(exp[1]))


def test_secp256k1_adapter_callback():
    n = 40
    rnd = random.Random(8)
    pts = rand_points(SE, n, 77)
    pts[3] = None
    sc = [rnd.randrange(SE.n) for _ in range(n)]
    sc[5] = 0
    ok, res = pb.secp256k1_ecmult_multi_var(sc, pts, g_scalar=0)
    assert ok == 1 and res == O.msm(SE, sc, pts)
    ok, res = pb.secp256k1_ecmult_multi_var(sc, pts, g_scalar=12345)
    assert res == O.add(SE, O.msm(SE, sc, pts), O.mul(SE, 12345, (SE.gx, SE.gy)))
    ok, res = pb.secp256k1_ecmult_multi_var([], [], g_scalar=None)
    assert ok == 1 and res is None


def test_secp256k1_adapter_edge_cases_of_the_reference_suite():
    """The shapes of test_ecmult_multi (/root/reference/porla/Utils/secp256k1_lib/tests.c:3816-4053) through
    the adapter: cancelling pairs, all-infinity, all-zero scalars, constant scalar, constant point, scalars
    >= n (convert_ZZ_to_scalar does not reduce, utils.h:180-192), a failing callback."""
    rnd = random.Random(31)
    G = (SE.gx, SE.gy)
    P, Q = O.mul(SE, 0x1234567, G), O.mul(SE, 0x7654321, G)
    run = pb.secp256k1_ecmult_multi_var
    # sc*P + (-sc)*P, and sc*P + sc*(-P)
    sc = rnd.randrange(SE.n)
    assert run([sc, SE.n - sc], [P, P], 0) == (1, None)
    assert run([sc, sc], [P, O.neg(SE, P)], 0) == (1, None)
    # all-infinity points / all-zero scalars, sizes straddling the reference's Strauss/Pippenger switch (88)
    for n in (1, 2, 32, 88, 130):
        assert run([rnd.randrange(SE.n) for _ in range(n)], [None] * n, 0) == (1, None)
        assert run([0] * n, [O.mul(SE, i + 1, G) for i in range(n)], 0) == (1, None)
    # constant scalar over many points, constant point under many scalars
    n = 100
    pts = [O.mul(SE, rnd.randrange(1, 1 << 64), G) for _ in range(n)]
    assert run([sc] * n, pts, 0) == (1, O.mul(SE, sc, O.msm(SE, [1] * n, pts)))
    scs = [rnd.randrange(SE.n) for _ in range(n)]
    assert run(scs, [Q] * n, 0) == (1, O.mul(SE, sum(scs) % SE.n, Q))
    # unreduced scalars
    big = [SE.n + 5, (1 << 256) - 1, SE.n]
    assert run(big, [P, Q, P], 0) == (1, O.msm(SE, [s % SE.n for s in big], [P, Q, P]))
    # a callback that fails makes the call return 0 (ecmult_impl.h:700-703)
    lib = pb.load()
    from porla_b200.lib import SECP_CB, SecpGej
    r = SecpGej()
    ok = lib.porla_secp256k1_ecmult_multi_var(None, None, C.byref(r), None, SECP_CB(lambda s, p, i, d: 0), None, 4)
    assert ok == 0 and r.infinity == 1


def test_secp256k1_resident_generators():
    """Generators uploaded once (porla_secp256k1_table_create), MSMs over sub-ranges with host scalars: the
    call shape of Porla's IPA commitments (data.pt = &generators[start_chunk], Server.hpp:347)."""
    rnd = random.Random(99)
    G = (SE.gx, SE.gy)
    gens = [O.mul(SE, rnd.randrange(1, SE.n), G) for _ in range(130)]
    gens[7] = None
    tab = pb.SecpGenerators(gens)
    for first, n in ((0, 130), (3, 40), (16, 16), (100, 30), (7, 1), (129, 1)):
        sc = [rnd.randrange(1 << 256) for _ in range(n)]
        if n > 4:
            sc[2] = 0
        ok, res = tab.multi(first, sc)
        assert ok == 1 and res == O.msm(SE, [s % SE.n for s in sc], gens[first:first + n]), (first, n)
    assert tab.multi(0, []) == (1, None)
    assert tab.multi(120, [1] * 20)[0] == 0                    # leaves the table
    # same answer as the callback adapter
    sc = [rnd.randrange(SE.n) for _ in range(64)]
    assert tab.multi(32, sc)[1] == pb.secp256k1_ecmult_multi_var(sc, gens[32:96], g_scalar=0)[1]
    tab.destroy()
