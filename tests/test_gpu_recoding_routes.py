"""The radix-sort route of a single MSM (2^19 terms or more) at every window layout it accepts, with scalars on the edges
of the signed-digit recoding, against closed forms.

That route recodes each scalar twice, in k_coarse_count (a 64-bit shift register over the limbs) and in
k_partition_coarse (funnel shifts over the tile's words in shared memory, carries kept in registers across windows), and
both must agree with k_digits, which the atomic-scatter sort and every smaller MSM use.  A wrong digit still yields a
valid point, so every result here is compared with a closed form: the table is P_i = k_i G with k_i < 2^31 (some 0:
infinity), each scalar family draws from a pool of a few thousand values, and MSM(s) = [sum_v v K_v] G with K_v the sum
of the k_i of the terms that carry value v (exact in int64).  oracle/recoding_py.py restates the recoding and builds the
families.

Routes at n = 2^19 + 37, from the conditions in msm_impl.cuh (radix: at most 28 windows; sort_v2: at most 0.95 kBigBin
pairs per coarse bin on average; k_reduce above 600 k buckets on BN254, 300 k on secp256k1):

    layout                                        sort                                              reduction
    c = 9, every curve and split                  atomic scatter, 2 launches (29 or 30 windows)     quad scan + top
    BN254 plain, c = 10                           sort_v2; its top window (4 bits + carry) puts      quad scan + top
                                                  all n pairs into one coarse bin: big-bin route
    BN254 GLV, c = 10                             exact histogram + radix (65 540 pairs per bin)    quad scan + top
    BN254 plain 11-16, GLV 11-17, secp256k1 10-14 sort_v2                                           quad scan + top
    secp256k1, c = 15                             sort_v2; the top window holds only the carry      quad scan + top
    secp256k1, c = 17                             sort_v2; the top window holds only the carry      k_reduce
    BN254 plain 17-20, GLV 18-20, secp256k1 16-20 sort_v2                                           k_reduce

PORLA_SORT_V2=0 / 1 and PORLA_ATOMIC_SCATTER=1 move every radix layout to the other sorts; the first 2^19 - 1 terms of
the same scalars take the atomic scatter, which emits 16 windows per launch and recomputes the carries of the windows it
skips (two launches whenever there are more than 16 windows).
"""
import ctypes as C

import numpy as np
import pytest

import porla_b200 as pb
from oracle import curves_py as O
from oracle import recoding_py as R

pytestmark = pytest.mark.gpu

N = (1 << 19) + 37
PREFIX = (1 << 19) - 1
POOL = 1024                                  # distinct values per family ('mixed': all of them, about 4 to 5 k)
CURVES = {pb.CURVE_BN254: O.BN254, pb.CURVE_SECP256K1: O.SECP256K1}
LAYOUTS = [(curve, glv, c) for curve in CURVES for glv in ((False, True) if curve == pb.CURVE_BN254 else (False,))
           for c in range(9, 21)]
ROUTES = {"default": {}, "sort_v2=0": {"PORLA_SORT_V2": "0"}, "sort_v2=1": {"PORLA_SORT_V2": "1"},
          "atomic_scatter": {"PORLA_ATOMIC_SCATTER": "1"}}
SWITCHES = ("PORLA_SORT_V2", "PORLA_ATOMIC_SCATTER")


def _layout_id(curve, glv, c):
    return "%s-%s-c%d" % ("bn254" if curve == pb.CURVE_BN254 else "secp256k1", "glv" if glv else "plain", c)


def _code(glv, c):
    return c | (pb.lib.PLAN_GLV_ON if glv else pb.lib.PLAN_GLV_OFF)


@pytest.fixture(scope="module")
def tables():
    """One table per curve: P_i = k_i G, k_i < 2^31, every 97th k_i = 0 (infinity points the recoders drop)."""
    import torch
    rng = np.random.default_rng(2019)
    out = {}
    for curve in CURVES:
        ks = rng.integers(1, 1 << 31, size=N, dtype=np.int64)
        ks[3::97] = 0
        limbs = np.zeros((N, 8), np.uint32)
        limbs[:, 0] = ks
        d_ks = torch.from_numpy(limbs.view(np.int32)).cuda()
        tab = pb.Table.multiples_of_generator(curve, d_ks.data_ptr(), N, pb.SCALAR_LE32, on_device=True)
        assert tab.num_infinity == int((ks == 0).sum())
        out[curve] = (tab, ks.astype(np.float64))
    yield out
    for tab, _ in out.values():
        tab.destroy()


class Case:
    """One scalar family spread over the N terms by index, uploaded in BE32 or LE32."""

    def __init__(self, pool, seed, fmt, ks):
        import torch
        self.pool, self.fmt = pool, fmt
        self.assign = np.random.default_rng(seed).integers(0, len(pool), size=N)
        order = "big" if fmt == pb.SCALAR_BE32 else "little"
        raw = np.frombuffer(b"".join(v.to_bytes(32, order) for v in pool), np.uint8).reshape(len(pool), 32)
        self.d_sc = torch.from_numpy(raw[self.assign]).cuda()
        self.ks = ks

    def group_sums(self, m):
        """K_v over the first m terms: sums of fewer than 2^20 values below 2^31, exact in float64."""
        return [int(k) for k in np.rint(np.bincount(self.assign[:m], weights=self.ks[:m], minlength=len(self.pool)))]

    def total(self, curve, m):
        return sum(v * k for v, k in zip(self.pool, self.group_sums(m))) % curve.n


def _enc(P):
    return bytes(64) if P is None else P[0].to_bytes(32, "big") + P[1].to_bytes(32, "big")


def _route_env(monkeypatch, env):
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


@pytest.mark.parametrize("curve,glv,c", LAYOUTS, ids=[_layout_id(*l) for l in LAYOUTS])
def test_every_route_matches_the_closed_form(tables, curve, glv, c, monkeypatch):
    """Each family at this forced layout through the default route, both radix sorts, the atomic scatter and the
    2^19 - 1-term prefix: every result equals [sum_i s_i k_i] G."""
    tab, ks = tables[curve]
    cv = CURVES[curve]
    G = (cv.gx, cv.gy)
    code = _code(glv, c)
    failures = []
    fams = R.families(cv, glv, c, POOL, seed=1000 * curve + 100 * glv + c)
    for i, (name, pool) in enumerate(fams.items()):
        case = Case(pool, seed=i + 7 * c, fmt=pb.SCALAR_BE32 if (c + i) % 2 == 0 else pb.SCALAR_LE32, ks=ks)
        want = _enc(O.mul(cv, case.total(cv, N), G))
        for route, env in ROUTES.items():
            _route_env(monkeypatch, env)
            if tab.msm_resident(case.d_sc.data_ptr(), N, scalar_fmt=case.fmt, window_bits=code) != want:
                failures.append((name, route))
        _route_env(monkeypatch, {})
        want = _enc(O.mul(cv, case.total(cv, PREFIX), G))
        if tab.msm_resident(case.d_sc.data_ptr(), PREFIX, scalar_fmt=case.fmt, window_bits=code) != want:
            failures.append((name, "prefix 2^19 - 1"))
    assert not failures, "%s: (family, route) off the closed form: %s" % (_layout_id(curve, glv, c), failures)


def _xyzz_affine(cv, rec):
    """128-byte XYZZ record (X, Y, ZZ, ZZZ as little-endian limbs, in the field's internal form) -> affine or None.
    x = X / ZZ and y = Y / ZZZ: the ratios cancel the Montgomery factor."""
    X, Y, ZZ, ZZZ = (int.from_bytes(rec[32 * j:32 * j + 32], "little") % cv.p for j in range(4))
    if ZZ == 0:
        return None
    return X * pow(ZZ, -1, cv.p) % cv.p, Y * pow(ZZZ, -1, cv.p) % cv.p


# one layout per row of the route table
WINDOW_LAYOUTS = [(pb.CURVE_BN254, True, 9), (pb.CURVE_BN254, False, 10), (pb.CURVE_BN254, True, 10),
                  (pb.CURVE_SECP256K1, False, 13), (pb.CURVE_SECP256K1, False, 15), (pb.CURVE_SECP256K1, False, 17),
                  (pb.CURVE_BN254, False, 17), (pb.CURVE_BN254, True, 19)]


@pytest.mark.parametrize("curve,glv,c", WINDOW_LAYOUTS, ids=[_layout_id(*l) for l in WINDOW_LAYOUTS])
def test_window_sums_match_the_recoding(tables, curve, glv, c, monkeypatch):
    """Window slot w's sum over every route equals [sum_i delta_w(s_i) k_i] G, delta_w from the restated recoding
    (sign * d; sign1 * d1 + sign2 * d2 * lambda with GLV): a wrong digit is pinned to its window."""
    import torch
    tab, ks = tables[curve]
    cv = CURVES[curve]
    G = (cv.gx, cv.gy)
    code = _code(glv, c)
    cc, nwin = C.c_int(0), C.c_int(0)
    pb.load().porla_msm_plan(curve, N, 1, code, C.byref(cc), C.byref(nwin))
    assert cc.value == code and nwin.value == R.num_windows(cv, glv, c)
    nwin = nwin.value
    d_w = torch.zeros(nwin * 128, dtype=torch.uint8, device="cuda")

    def window_sums(case, n):
        pb.load().porla_msm_window_sums_device(C.c_void_p(tab.handle), C.c_void_p(case.d_sc.data_ptr()), n, case.fmt, code,
                                               C.c_void_p(d_w.data_ptr()), None)
        torch.cuda.synchronize()
        raw = d_w.cpu().numpy().tobytes()
        return [_xyzz_affine(cv, raw[128 * w:128 * w + 128]) for w in range(nwin)]

    failures = []
    fams = R.families(cv, glv, c, POOL, seed=31 * c + glv)
    for i, (name, pool) in enumerate(fams.items()):
        case = Case(pool, seed=100 + i, fmt=pb.SCALAR_LE32 if (c + i) % 2 == 0 else pb.SCALAR_BE32, ks=ks)
        deltas = [R.window_multipliers(cv, glv, c, v) for v in pool]
        want = {}
        for m in (N, PREFIX):
            K = case.group_sums(m)
            want[m] = [O.mul(cv, sum(d[w] * k for d, k in zip(deltas, K)) % cv.n, G) for w in range(nwin)]
        runs = [(route, env, N) for route, env in ROUTES.items()] + [("prefix 2^19 - 1", {}, PREFIX)]
        for route, env, m in runs:
            _route_env(monkeypatch, env)
            got = window_sums(case, m)
            bad = [w for w in range(nwin) if got[w] != want[m][w]]
            if bad:
                failures.append("%s / %s: windows %s" % (name, route, bad))
        _route_env(monkeypatch, {})
    assert not failures, "%s, window sums off the recoding: %s" % (_layout_id(curve, glv, c), "; ".join(failures))
