"""The IPA-mode server entries (porla_secp256k1_align_mac_batch, porla_secp256k1_audit_aggregate,
porla_secp256k1_ecmult_multi_gej) at their boundary: refused shapes return 0 and leave every buffer as it was, and empty
calls answer without initialising a device (these tests carry no gpu mark, so they also run where there is none)."""
import ctypes as C
import random

import pytest

import porla_b200 as pb
from oracle import curves_py as O
from tests.test_secp_butterfly import SE, G, to_gej


def _align_buffers(batch, n_chunks):
    rnd = random.Random(batch * 1000 + n_chunks)
    data = bytearray(rnd.randbytes(64 * max(1, batch * n_chunks)))
    out = (pb.lib.SecpGej * max(1, batch))()
    C.memmove(out, rnd.randbytes(C.sizeof(out)), C.sizeof(out))
    return data, out


@pytest.mark.parametrize("n_chunks,batch", [(128, 1), (128, 0), (0, 4), (1, 1)])
def test_align_without_a_table_is_refused(n_chunks, batch):
    lib = pb.load()
    data, out = _align_buffers(batch, n_chunks)
    before = (bytes(data), bytes(out))
    assert lib.porla_secp256k1_align_mac_batch(None, n_chunks, pb.lib._as_void_p(data), batch, out) == 0
    assert (bytes(data), bytes(out)) == before


@pytest.mark.parametrize("n", [0, 1, 766, 1 << 24])
def test_audit_without_a_table_is_refused(n):
    lib = pb.load()
    rnd = random.Random(n)
    coefs = bytearray(rnd.randbytes(4 * min(n, 766) + 4))
    blocks = bytearray(rnd.randbytes(64 * 4))
    b_out = bytearray(rnd.randbytes(32 * 4))
    al = pb.lib.SecpGej()
    C.memmove(C.byref(al), rnd.randbytes(C.sizeof(al)), C.sizeof(al))
    before = (bytes(coefs), bytes(blocks), bytes(b_out), bytes(al))
    assert lib.porla_secp256k1_audit_aggregate(None, 4, pb.lib._as_void_p(coefs), pb.lib._as_void_p(blocks), n,
                                               pb.lib._as_void_p(b_out), C.byref(al)) == 0
    assert (bytes(coefs), bytes(blocks), bytes(b_out), bytes(al)) == before


@pytest.mark.parametrize("n,nbatch", [(1 << 31, 1), (1 << 30, 2), (3, 1 << 30), (1 << 62, 4)])
def test_gej_multi_exponentiation_past_32_bit_terms_is_refused(n, nbatch):
    """n * nbatch >= 2^31 terms: refused before any input is read (the arrays passed are far shorter)."""
    rnd = random.Random(n ^ nbatch)
    pts = to_gej([O.mul(SE, 3, G), None], rnd)
    sc = (pb.lib.SecpScalar * 2)()
    r = (pb.lib.SecpGej * 4)()
    C.memmove(r, rnd.randbytes(C.sizeof(r)), C.sizeof(r))
    before = (bytes(pts), bytes(sc), bytes(r))
    assert pb.load().porla_secp256k1_ecmult_multi_gej(pts, sc, n, nbatch, r) == 0
    assert (bytes(pts), bytes(sc), bytes(r)) == before


@pytest.mark.parametrize("n,nbatch", [(0, 1), (0, 5), (7, 0), (0, 0)])
def test_empty_gej_multi_exponentiation_needs_no_device(n, nbatch):
    """Nothing to multiply: every result is infinity as gej_set_infinity writes it, and no device is initialised."""
    rnd = random.Random(n + 10 * nbatch)
    pts = to_gej([O.mul(SE, 5 + i, G) for i in range(max(1, n * nbatch))], rnd)
    ok, r = pb.secp256k1_ecmult_multi_gej(pts, [rnd.randrange(SE.n) for _ in range(n * nbatch)], n, nbatch)
    assert ok == 1
    for g in r[:nbatch]:
        assert g.infinity == 1
        assert [list(g.x.n), list(g.y.n), list(g.z.n)] == [[0] * 5] * 3
