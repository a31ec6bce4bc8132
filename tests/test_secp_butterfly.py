"""secp256k1 butterflies of the FFT in the exponent (IPA mode): the endomorphism constants of ec.cuh, the rounded split
they feed, and the host route of porla_secp256k1_butterfly_stage (small stages never touch the device)."""
import os
import random
import re

import pytest

import porla_b200 as pb
from oracle import curves_py as O

SE = O.SECP256K1
G = (SE.gx, SE.gy)
EC_CUH = os.path.join(os.path.dirname(__file__), "..", "porla_b200", "csrc", "ec.cuh")


def _secp_constant(name):
    src = open(EC_CUH).read()
    body = src[src.index("struct Secp256k1 {"):]
    vals = re.search(r"%s\(int i\) \{[^}]*?m\[\d+\] = \{([^}]*)\}" % name, body, re.S).group(1)
    return sum(int(v.strip().rstrip("u"), 16) << (32 * i) for i, v in enumerate(vals.split(",")))


def split_oracle(k, g=None):
    """glv_split_secp256k1 (ec.cuh) restated: c1, c2 rounded at bit 383 of k * g1, k * g2."""
    g = g or O.glv_constants(SE)
    g1, g2 = _secp_constant("glv_g1"), _secp_constant("glv_g2")
    c1 = (k * g1 >> 384) + (k * g1 >> 383 & 1)
    c2 = (k * g2 >> 384) + (k * g2 >> 383 & 1)
    return k - c1 * g["a1"] - c2 * g["a2"], -c1 * g["b1"] - c2 * g["b2"]


def test_secp256k1_endomorphism_constants_in_the_kernel_header():
    """Secp256k1::glv_* against cube roots of unity mod p and mod n and the extended-Euclid basis (curves_py.glv_constants)."""
    g = O.glv_constants(SE)
    assert pow(g["beta"], 3, SE.p) == 1 and pow(g["lambda"], 3, SE.n) == 1
    assert O.mul(SE, g["lambda"], G) == (g["beta"] * SE.gx % SE.p, SE.gy)
    assert _secp_constant("glv_beta_mont") == g["beta"]          # the field is kept plain: internal form = beta
    assert _secp_constant("glv_lambda") == g["lambda"]
    assert _secp_constant("glv_g1") == ((g["b2"] << 384) + SE.n // 2) // SE.n
    assert _secp_constant("glv_g2") == (((-g["b1"]) << 384) + SE.n // 2) // SE.n
    assert _secp_constant("glv_a1") == g["a1"] == g["b2"] == 0x3086D221A7D46BCDE86C90E49284EB15
    assert _secp_constant("glv_nb1") == -g["b1"] == 0xE4437ED6010E88286F547FA90ABFE4C3
    assert _secp_constant("glv_a2") == g["a2"] == 0x114CA50F7A8E2F3F657C1108D9D44CFD8
    assert g["a1"] * g["b2"] - g["a2"] * g["b1"] == SE.n


def test_secp256k1_rounded_split_is_exact_and_within_128_bits():
    g = O.glv_constants(SE)
    lam, n = g["lambda"], SE.n
    rnd = random.Random(2024)
    corners = [0, 1, 2, n - 1, n - 2, n // 2, n // 2 + 1, lam, n - lam, (1 << 128) - 1, 1 << 128, 1 << 255, n - (1 << 128)]
    corners += [(i * lam + j) % n for i in (-1, 0, 1) for j in ((1 << 127), (1 << 128) - 1, -(1 << 127))]
    worst = 0
    for k in corners + [rnd.randrange(n) for _ in range(200000)]:
        k1, k2 = split_oracle(k, g)
        assert (k1 + k2 * lam - k) % n == 0, hex(k)
        assert abs(k1) < 1 << 128 and abs(k2) < 1 << 128, hex(k)
        worst = max(worst, abs(k1), abs(k2))
    assert worst >= 1 << 127          # the bound is tight: the quad kernel's 64 two-bit digits are all used


# ---------------------------------------------------------------------------- host-buffer entry
def butterfly_oracle(pts, m, tw):
    """The loop body of Server.hpp:1577-1608 (secp256k1_ecmult + 2 gej_add_var in IPA mode) for every butterfly."""
    out = list(pts)
    m2 = m // 2
    for j in range(m2):
        for k in range(j, len(pts), m):
            t = O.mul(SE, tw[j] % SE.n, pts[k + m2])
            out[k] = O.add(SE, pts[k], t)
            out[k + m2] = O.add(SE, pts[k], O.neg(SE, t))
    return out


def _fe_loose(v, rnd):
    """v (< p) as 5 x 52-bit limbs of v + j p with some weight moved down a limb: a field element of magnitude > 1."""
    w = v + rnd.randrange(4) * SE.p
    limbs = [(w >> (52 * i)) & ((1 << 52) - 1) for i in range(4)] + [w >> 208]
    for i in range(4):
        d = min(limbs[i + 1], rnd.randrange(1 << 8))
        limbs[i + 1] -= d
        limbs[i] += d << 52
    assert sum(l << (52 * i) for i, l in enumerate(limbs)) == w
    fe = pb.lib.SecpFe()
    for i, l in enumerate(limbs):
        fe.n[i] = l
    return fe


def to_gej(pts, rnd, z_one=False):
    """Affine points (None = infinity) -> a ctypes array of SecpGej with random z != 1 and non-normalised limbs."""
    arr = (pb.lib.SecpGej * len(pts))()
    for i, P in enumerate(pts):
        if P is None:
            arr[i].infinity = 1
            arr[i].x = _fe_loose(rnd.randrange(SE.p), rnd)     # garbage coordinates must be ignored
            continue
        z = 1 if z_one else rnd.randrange(2, SE.p)
        arr[i].x = _fe_loose(P[0] * z * z % SE.p, rnd)
        arr[i].y = _fe_loose(P[1] * pow(z, 3, SE.p) % SE.p, rnd)
        arr[i].z = _fe_loose(z, rnd)
        arr[i].infinity = 0
    return arr


def from_gej(arr):
    """Outputs as the entry promises them: z = 1, normalised limbs, infinity as gej_set_infinity writes it."""
    out = []
    for g in arr:
        limbs = [list(g.x.n), list(g.y.n), list(g.z.n)]
        if g.infinity:
            assert g.infinity == 1 and limbs == [[0] * 5] * 3
            out.append(None)
            continue
        for fe in limbs:
            assert all(l < 1 << 52 for l in fe[:4]) and fe[4] < 1 << 48
        assert limbs[2] == [1, 0, 0, 0, 0]
        x, y = (sum(l << (52 * i) for i, l in enumerate(fe)) for fe in limbs[:2])
        assert x < SE.p and y < SE.p
        out.append((x, y))
    return out


def long_half_scalars(count, seed):
    """Twiddles whose split halves reach 2^127 ... 2^128."""
    rnd, g, out = random.Random(seed), O.glv_constants(SE), []
    while len(out) < count:
        k = rnd.randrange(SE.n)
        if max(abs(h) for h in split_oracle(k, g)) >= 1 << 127:
            out.append(k)
    return out


def edge_case_stage(seed):
    """One stage of n = 16, m = 8: twiddle j serves the butterflies (j, j + 4) and (j + 8, j + 12)."""
    rnd = random.Random(seed)
    n, m = 16, 8
    pts = [O.mul(SE, rnd.randrange(1, SE.n), G) for _ in range(n)]
    tw = [0, 1, SE.n - 1, SE.n + 5]                 # 0, 1, n - 1 and one >= n (taken mod n)
    pts[4] = None                                   # A1 = infinity
    pts[1] = None                                   # A0 = infinity
    pts[9] = pts[13]                                # A0 = t  (w = 1): P[k] - t is infinity
    pts[10] = pts[14]                               # A0 = -t (w = n - 1): P[k] + t is infinity
    pts[11] = O.mul(SE, 5, pts[15])                 # A0 = t  (w = n + 5)
    return pts, m, tw


def long_half_stage(seed):
    rnd = random.Random(seed)
    n, m = 16, 16
    pts = [O.mul(SE, rnd.randrange(1, SE.n), G) for _ in range(n)]
    return pts, m, long_half_scalars(m // 2, seed)


@pytest.mark.parametrize("case", [edge_case_stage, long_half_stage], ids=["edges", "long_halves"])
def test_host_route_matches_oracle(case, monkeypatch):
    monkeypatch.setenv("PORLA_HOST_BUTTERFLIES", "1000000")
    pts, m, tw = case(11)
    rnd = random.Random(3)
    arr = to_gej(pts, rnd)
    assert pb.secp256k1_butterfly_stage(arr, m, tw) == 1
    assert from_gej(arr) == butterfly_oracle(pts, m, tw)


def test_host_route_full_transform_on_its_own_outputs(monkeypatch):
    """log2 n stages, each on the previous stage's outputs (z = 1 from the second stage on)."""
    monkeypatch.setenv("PORLA_HOST_BUTTERFLIES", "1000000")
    rnd = random.Random(8)
    n = 16
    cur = [O.mul(SE, rnd.randrange(1, SE.n), G) for _ in range(n)]
    cur[3] = None
    arr = to_gej(cur, rnd)
    m = 2
    while m <= n:
        tw = [rnd.randrange(1 << 256) for _ in range(m // 2)]
        assert pb.secp256k1_butterfly_stage(arr, m, tw) == 1
        cur = butterfly_oracle(cur, m, tw)
        assert from_gej(arr) == cur
        m *= 2


@pytest.mark.parametrize("n,m", [(16, 3), (16, 32), (12, 8), (16, 0), (16, 1)])
def test_bad_stage_shape_is_refused_and_leaves_the_buffer(n, m):
    rnd = random.Random(n + m)
    arr = to_gej([O.mul(SE, i + 1, G) for i in range(n)], rnd)
    before = bytes(arr)
    assert pb.secp256k1_butterfly_stage(arr, m, [1] * max(1, m // 2)) == 0
    assert bytes(arr) == before
