"""The MSM engine's signed-digit recoding, restated with Python integers, and scalar families that sit on its edges.

TEST INFRASTRUCTURE ONLY (see curves_py).  The device has three recoders that must agree digit for digit: k_digits
(small and batched MSMs, and the atomic-scatter sort), k_coarse_count and k_partition_coarse (the radix sort of a single
MSM of 2^19 terms or more), all in porla_b200/csrc/msm_kernels.cuh.  What they compute for a scalar s (any 256-bit
integer, read as BE32 or LE32):

* s is reduced mod the group order.  secp256k1 recodes min(s, n - s) and negates the point when it took n - s.  BN254
  with the GLV split recodes the two halves |k1|, |k2| < 2^127 of s = k1 + k2 lambda (curves_py.glv_split), each with
  the sign of its half; window w of both halves fills the buckets of window slot w, the second half with phi(P) = lambda P.
* A value v is cut into nwin windows of c bits, nwin = ceil((bits + 1) / c) with bits = 254 (BN254), 255 (secp256k1
  after the flip) or 127 (a GLV half).  Window w has the raw digit (v >> c w) mod 2^c plus the carry out of window w - 1;
  a digit d > 2^(c-1) becomes d - 2^c and carries 1 into window w + 1.  A digit of exactly 2^(c-1) stays positive.
  |d| - 1 is the bucket, the sign of d (times the sign of the half) the sign of the point.

So the pairs of scalar s put delta_w(s) P into the buckets of window slot w, and the window sum of slot w over the
terms (s_i, P_i = k_i G) is [sum_i delta_w(s_i) k_i] G: the per-window closed form the tests check.
"""
from __future__ import annotations

import functools
import random

from oracle import curves_py as O

BN, SE = O.BN254, O.SECP256K1
SCALAR_BITS = {BN.name: 254, SE.name: 255}   # r < 2^254; the secp256k1 magnitude min(s, n - s) < 2^255
GLV_BITS = 127


@functools.lru_cache(maxsize=None)
def glv_consts():
    return O.glv_constants(BN)


def num_windows(curve, glv: bool, c: int) -> int:
    """Windows per scalar (per half with GLV): the value's bits plus the carry of the top digit, as msm_plan counts them."""
    bits = GLV_BITS if glv else SCALAR_BITS[curve.name]
    return (bits + 1 + c - 1) // c


def signed_digits(v: int, c: int, nwin: int):
    """Signed c-bit digits of v >= 0, low window first, and the carry out of the top window."""
    half, mask = 1 << (c - 1), (1 << c) - 1
    digits, carry = [], 0
    for w in range(nwin):
        d = ((v >> (c * w)) & mask) + carry
        carry = 1 if d > half else 0
        digits.append(d - (carry << c))
    return digits, carry


def halves(curve, glv: bool, s: int):
    """[(sign, magnitude)] of the values the recoder walks for scalar s: one, or the two GLV halves."""
    s %= curve.n
    if glv:
        k1, k2 = O.glv_split(curve, s, glv_consts())
        return [(-1 if k1 < 0 else 1, abs(k1)), (-1 if k2 < 0 else 1, abs(k2))]
    if curve is SE and curve.n - s < s:
        return [(-1, curve.n - s)]
    return [(1, s)]


def recode(curve, glv: bool, c: int, s: int):
    """[(sign, digits, carry out of the top window)] per half."""
    nwin = num_windows(curve, glv, c)
    return [(sign, *signed_digits(v, c, nwin)) for sign, v in halves(curve, glv, s)]


def window_multipliers(curve, glv: bool, c: int, s: int):
    """delta_w(s) mod the order for every window slot w: sign * d, or sign1 * d1 + sign2 * d2 * lambda with GLV."""
    lam = glv_consts()["lambda"] if glv else 0
    out = [0] * num_windows(curve, glv, c)
    for h, (sign, digits, _) in enumerate(recode(curve, glv, c, s)):
        f = sign * (lam if h else 1)
        for w, d in enumerate(digits):
            out[w] += f * d
    return [x % curve.n for x in out]


# --------------------------------------------------------------------------- scalar families
# Each returns `count` distinct-ish scalars (Python ints below 2^256) for the window layout (curve, glv, c).
def _magnitude_bound(curve, glv: bool) -> int:
    """Largest magnitude the family builders aim at: r - 1, (n - 1) / 2 (no flip), or a2 for a GLV half (the floor split
    returns halves up to about a2 < 2^127; glv_split decides which candidates it really returns)."""
    if glv:
        return glv_consts()["a2"]
    return BN.n - 1 if curve is BN else (SE.n - 1) // 2


def _with_digits(rnd: random.Random, c: int, bound: int, digit) -> int:
    """A value <= bound whose c-bit windows below the top one all hold the raw digit digit(rnd).  Three in four are as
    long as `bound`, the others shorter (their top digits are zero)."""
    if rnd.random() < 0.25:
        bound = min(bound, (1 << rnd.randrange(c + 1, bound.bit_length() + 1)) - 1)
    nw = (bound.bit_length() - 1) // c                 # windows wholly below the top bit of bound
    low = sum(digit(rnd) << (c * w) for w in range(nw))
    return low + (rnd.randrange(bound >> (c * nw)) << (c * nw))


def _unreduced(rnd: random.Random, curve, s: int) -> int:
    """s plus a random multiple of the order that keeps it below 2^256 (the recoders reduce first)."""
    j = rnd.randrange(((1 << 256) - 1 - s) // curve.n + 1)
    return s + j * curve.n


def _from_magnitudes(rnd: random.Random, curve, glv: bool, c: int, count: int, digit):
    out = []
    if glv:
        g, r = glv_consts(), BN.n
        bound = _magnitude_bound(curve, True)
        while len(out) < count:
            k1 = _with_digits(rnd, c, bound, digit)
            k2 = -_with_digits(rnd, c, bound, digit) if rnd.random() < 0.85 else 0
            s = (k1 + k2 * g["lambda"]) % r
            if O.glv_split(BN, s, g) == (k1, k2):       # halves the split really produces
                out.append(_unreduced(rnd, curve, s) if rnd.random() < 0.5 else s)
        return out
    bound = _magnitude_bound(curve, False)
    while len(out) < count:
        t = _with_digits(rnd, c, bound, digit)
        if curve is SE:
            out.append(SE.n - t if rnd.random() < 0.5 else t)  # above n / 2: recoded as -(n - s), magnitude t again
        else:
            out.append(_unreduced(rnd, curve, t) if rnd.random() < 0.5 else t)
    return out


def tie(curve, glv, c, count, rnd):
    """Raw digit 2^(c-1) in every window below the top: the last bucket of each window, kept positive, no carry."""
    half = 1 << (c - 1)
    return _from_magnitudes(rnd, curve, glv, c, count, lambda _r: half)


def carry_chain(curve, glv, c, count, rnd):
    """Raw digits 2^(c-1) + 1 or 2^c - 1: every window below the top goes negative (or to 0 with the carry, for 2^c - 1
    after a carry) and the carry runs from window 0 into the top window."""
    half = 1 << (c - 1)
    return _from_magnitudes(rnd, curve, glv, c, count, lambda r: half + 1 if r.random() < 0.5 else 2 * half - 1)


def uniform256(curve, glv, c, count, rnd):
    """Uniform 256-bit values: most of them above r on BN254, half of them above n / 2 on secp256k1."""
    return [rnd.getrandbits(256) for _ in range(count)]


def order_edges(curve, glv, c, count, rnd):
    """Values at the order and at the top-window boundaries of this layout, mixed with uniform ones."""
    o = curve.n
    vals = [0, 1, o - 1, o, o + 1, 2 * o - 1, 2 * o, 2 * o + 1, (1 << 256) - 1, (1 << 256) - o, (1 << 255) - 1, 1 << 255]
    if curve is SE:
        h = (o - 1) // 2                                 # (n - 1) / 2 is kept, (n + 1) / 2 is flipped to (n - 1) / 2
        vals += [h + d for d in range(-4, 6)] + [o - 2, 2 * h]
    else:
        vals += [j * o + d for j in range(3, 6) for d in (-1, 0, 1)]
    # the largest reduced value whose top window has each width, and the powers of two around it
    for k in range(max(1, c * (num_windows(curve, False, c) - 1) - c), 257):
        vals += [min((1 << k) - 1, o - 1), 1 << k, (1 << k) + 1]
    vals = [v for v in dict.fromkeys(vals) if 0 <= v < 1 << 256]
    return vals + uniform256(curve, glv, c, max(0, count - len(vals)), rnd)


@functools.lru_cache(maxsize=None)
def _largest_glv_halves(tries: int = 20000, keep: int = 24):
    """Host search: the scalars (of `tries` random ones) whose split has the largest max(|k1|, |k2|)."""
    rnd = random.Random(127)
    g = glv_consts()
    found = []
    for _ in range(tries):
        s = rnd.randrange(BN.n)
        k1, k2 = O.glv_split(BN, s, g)
        found.append((max(abs(k1), abs(k2)), s))
    return tuple(s for _, s in sorted(found, reverse=True)[:keep])


def glv_edges(curve, glv, c, count, rnd):
    """BN254 scalars at the corners of the GLV split.  The floor split never gives k1 < 0 (both floors round the lattice
    coordinates down), gives k2 < 0 for almost every scalar and k2 = 0 for scalars below about 2^126.8 (up to a2), so the corners are:
    the largest halves, k2 = 0, k1 = k2 = 0 (s = 0 and s = r), both halves near 2^127 (lambda, r - lambda), and
    all-ones magnitudes."""
    assert curve is BN
    g = glv_consts()
    lam, r = g["lambda"], BN.n
    vals = list(_largest_glv_halves()) + [0, r, 1, 2, (1 << 126) - 1, 1 << 126, g["a2"], g["a2"] - 1, -g["b1"]]
    vals += [lam, lam - 1, lam + 1, r - lam, r - lam + 1, r - 1, r + lam, (1 << 127) - 1, 1 << 127]
    ones = (1 << 126) - 1
    vals += [(ones + k2 * lam) % r for k2 in (-ones, -1, -(1 << 100))]
    vals = [v for v in dict.fromkeys(vals) if 0 <= v < 1 << 256]
    return vals + uniform256(curve, glv, c, max(0, count - len(vals)), rnd)


FAMILIES = {"uniform256": uniform256, "tie": tie, "carry_chain": carry_chain, "order_edges": order_edges, "glv_edges": glv_edges}


def families(curve, glv: bool, c: int, count: int, seed: int):
    """{name: scalars} for the layout, glv_edges only with GLV; 'mixed' is all the others together, and zeros."""
    rnd = random.Random(seed)
    out = {name: fn(curve, glv, c, count, rnd) for name, fn in FAMILIES.items() if name != "glv_edges" or glv}
    out["mixed"] = [0] * 16 + [v for vs in out.values() for v in vs]
    return out
