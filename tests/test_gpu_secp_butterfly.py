"""secp256k1 butterflies of the FFT in the exponent on the B200: porla_secp256k1_butterfly_stage on every route, a whole
transform through it, and resident tables at sizes that select each kernel, against the Python oracle and closed forms."""
import random

import pytest

import porla_b200 as pb
from oracle import curves_py as O
from tests.common import be, le
from tests.test_secp_butterfly import SE, G, butterfly_oracle, edge_case_stage, from_gej, long_half_scalars, long_half_stage, to_gej

ROUTES = {"host_threads": ("1000000", None), "quad": ("0", "1"), "one_thread": ("0", "0")}


@pytest.mark.gpu
@pytest.mark.parametrize("case", [edge_case_stage, long_half_stage], ids=["edges", "long_halves"])
@pytest.mark.parametrize("route", sorted(ROUTES))
def test_stage_matches_oracle_on_every_route(route, case, monkeypatch):
    host, quad = ROUTES[route]
    monkeypatch.setenv("PORLA_HOST_BUTTERFLIES", host)
    if quad is not None:
        monkeypatch.setenv("PORLA_BUTTERFLY_QUAD", quad)
    pts, m, tw = case(21)
    arr = to_gej(pts, random.Random(4))
    assert pb.secp256k1_butterfly_stage(arr, m, tw) == 1
    assert from_gej(arr) == butterfly_oracle(pts, m, tw)


@pytest.mark.gpu
def test_full_transform_of_256_macs_through_the_host_buffer_entry():
    """All 8 stages of n = 256 with the default routes (128 butterflies per stage: the device), inputs with random z."""
    rnd = random.Random(256)
    n = 256
    cur = [O.mul(SE, rnd.randrange(1, SE.n), G) for _ in range(n)]
    cur[7] = cur[200] = None
    arr = to_gej(cur, rnd)
    m = 2
    while m <= n:
        tw = [rnd.randrange(1 << 256) for _ in range(m // 2)]
        tw[0] = 0
        assert pb.secp256k1_butterfly_stage(arr, m, tw) == 1
        cur = butterfly_oracle(cur, m, tw)
        m *= 2
    assert from_gej(arr) == cur


def _transform(ks, m, tw):
    """The butterfly stage on the discrete logarithms: the transform is linear, so k_i G -> k'_i G."""
    out, m2 = list(ks), m // 2
    for j in range(m2):
        for k in range(j, len(ks), m):
            t = tw[j] * ks[k + m2]
            out[k], out[k + m2] = (ks[k] + t) % SE.n, (ks[k] - t) % SE.n
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n", [64, 1 << 15, 1 << 18], ids=["quad", "one_thread", "one_thread_full"])
def test_resident_table_stage_against_closed_form_then_msm(n):
    import torch

    rnd = random.Random(n)
    m = min(n, 1024)
    ks = [rnd.randrange(SE.n) for _ in range(n)]
    tw = [rnd.randrange(SE.n) for _ in range(m // 2 - 3)] + [0, 1, SE.n - 1]
    tw[1:1 + min(8, len(tw) - 4)] = long_half_scalars(min(8, len(tw) - 4), n)
    ks[5] = 0                                            # A0 = infinity
    ks[m // 2 + 9] = 0                                   # A1 = infinity
    ks[2] = tw[2] * ks[m // 2 + 2] % SE.n                # A0 = t: the second output is infinity
    ks[3] = -tw[3] * ks[m // 2 + 3] % SE.n               # A0 = -t: the first output is infinity
    t = pb.Table.multiples_of_generator(pb.CURVE_SECP256K1, b"".join(le(k) for k in ks), n)
    t.butterfly_stage(m, b"".join(be(w) for w in tw))
    got = t.export()
    want_ks = _transform(ks, m, tw)
    ref = pb.Table.multiples_of_generator(pb.CURVE_SECP256K1, b"".join(le(k) for k in want_ks), n)
    assert got == ref.export()
    ref.destroy()
    for i in sorted({2, 3, 5, m // 2 + 2, m // 2 + 3} | set(rnd.sample(range(n), 59))):
        P = O.mul(SE, want_ks[i], G) if want_ks[i] else None
        assert got[64 * i:64 * i + 64] == (bytes(64) if P is None else be(P[0]) + be(P[1])), i
    sc = [rnd.randrange(SE.n) for _ in range(n)]
    d_sc = torch.frombuffer(bytearray(b"".join(be(s) for s in sc)), dtype=torch.uint8).cuda()
    res = t.msm_resident(d_sc.data_ptr(), n)
    P = O.mul(SE, sum(s * k for s, k in zip(sc, want_ks)) % SE.n, G)
    assert res == (bytes(64) if P is None else be(P[0]) + be(P[1]))
    t.destroy()
