"""The IPA-mode client entries (porla_secp256k1_ecmult_const_batch, porla_secp256k1_ecmult_multi_table_batch) at their
boundary: refused shapes return 0 and leave every buffer as it was, and empty calls answer without initialising a device
(these tests carry no gpu mark, so they also run where there is none: a call that reached the device would abort there).

Without a device no table can be created, so the empty calls and the 2^31-term refusal run on a stand-in handle that
holds only what the entries read before they touch a device: the table's length and curve.  tests/test_gpu_ipa_client.py
checks that this layout matches a real table."""
import ctypes as C
import random

import pytest

import porla_b200 as pb


class TableHead(C.Structure):
    """The leading fields of porla_table (its PointTable, csrc/msm.h), padded past the end of the struct."""
    _fields_ = [("d_points", C.c_void_p), ("d_flags", C.c_void_p), ("n", C.c_uint32), ("n_inf", C.c_uint32),
                ("curve", C.c_int), ("rest", C.c_ubyte * 256)]


def stand_in(n, curve=pb.CURVE_SECP256K1):
    t = TableHead()
    t.n, t.curve = n, curve
    return t


def garbage(ctype, count, seed):
    """A ctypes array of `count` elements filled with random bytes (a buffer that must come back unchanged)."""
    arr = (ctype * max(1, count))()
    C.memmove(arr, random.Random(seed).randbytes(C.sizeof(arr)), C.sizeof(arr))
    return arr


def is_infinity(g):
    return g.infinity == 1 and [list(g.x.n), list(g.y.n), list(g.z.n)] == [[0] * 5] * 3


@pytest.mark.parametrize("n", [0, 1, 5, 1 << 31])
def test_complements_without_a_table_are_refused(n):
    sc, r = garbage(pb.lib.SecpScalar, min(n, 5), n), garbage(pb.lib.SecpGej, min(n, 5), n + 1)
    before = (bytes(sc), bytes(r))
    assert pb.load().porla_secp256k1_ecmult_const_batch(None, sc, n, r) == 0
    assert (bytes(sc), bytes(r)) == before


@pytest.mark.parametrize("table_len,curve,n", [(2, pb.CURVE_SECP256K1, 3), (0, pb.CURVE_SECP256K1, 3),
                                               (1, pb.CURVE_BN254, 3), (1, pb.CURVE_SECP256K1, 1 << 31),
                                               (1, pb.CURVE_SECP256K1, (1 << 64) - 1)])
def test_complements_on_a_bad_base_or_past_32_bit_counts_are_refused(table_len, curve, n):
    """A base whose length is not 1, a BN254 base, n >= 2^31: refused before any scalar is read (the arrays are far shorter)."""
    t = stand_in(table_len, curve)
    sc, r = garbage(pb.lib.SecpScalar, 3, n), garbage(pb.lib.SecpGej, 3, table_len)
    before = (bytes(t), bytes(sc), bytes(r))
    assert pb.load().porla_secp256k1_ecmult_const_batch(C.byref(t), sc, n, r) == 0
    assert (bytes(t), bytes(sc), bytes(r)) == before


def test_no_complements_need_no_device():
    t = stand_in(1)
    r = garbage(pb.lib.SecpGej, 1, 7)
    before = bytes(r)
    assert pb.load().porla_secp256k1_ecmult_const_batch(C.byref(t), None, 0, r) == 1
    assert bytes(r) == before


@pytest.mark.parametrize("n,batch", [(128, 1), (128, 0), (0, 4), (1 << 16, 1 << 15)])
def test_commitments_without_a_table_are_refused(n, batch):
    sc, r = garbage(pb.lib.SecpScalar, 8, n), garbage(pb.lib.SecpGej, 4, batch)
    before = (bytes(sc), bytes(r))
    assert pb.load().porla_secp256k1_ecmult_multi_table_batch(None, 0, sc, n, batch, r) == 0
    assert (bytes(sc), bytes(r)) == before


@pytest.mark.parametrize("table_len,curve,first,n,batch", [
    (0xFFFFFFFF, pb.CURVE_SECP256K1, 0, 1 << 16, 1 << 15),        # n * batch = 2^31
    (0xFFFFFFFF, pb.CURVE_SECP256K1, 0, 3, 1 << 30),
    (0xFFFFFFFF, pb.CURVE_SECP256K1, 5, (1 << 31) - 1, 2),
    (0xFFFFFFFF, pb.CURVE_SECP256K1, 0, 1, 1 << 31),
    (128, pb.CURVE_SECP256K1, 100, 29, 1),                        # first + n past the end
    (128, pb.CURVE_SECP256K1, 129, 0, 1),
    (128, pb.CURVE_SECP256K1, (1 << 64) - 1, 2, 1),               # first + n wraps around
    (128, pb.CURVE_BN254, 0, 128, 1),
])
def test_commitments_on_a_bad_table_or_range_are_refused(table_len, curve, first, n, batch):
    t = stand_in(table_len, curve)
    sc, r = garbage(pb.lib.SecpScalar, 8, n), garbage(pb.lib.SecpGej, 4, first)
    before = (bytes(t), bytes(sc), bytes(r))
    assert pb.load().porla_secp256k1_ecmult_multi_table_batch(C.byref(t), first, sc, n, batch, r) == 0
    assert (bytes(t), bytes(sc), bytes(r)) == before


@pytest.mark.parametrize("first,n,batch", [(0, 0, 1), (128, 0, 5), (3, 7, 0), (0, 0, 0)])
def test_empty_commitments_need_no_device(first, n, batch):
    """batch == 0 does nothing; n == 0 sets every r[b] to infinity as gej_set_infinity writes it."""
    t = stand_in(128)
    r = garbage(pb.lib.SecpGej, 6, first + batch)
    before = bytes(r)
    assert pb.load().porla_secp256k1_ecmult_multi_table_batch(C.byref(t), first, None, n, batch, r) == 1
    if batch == 0:
        assert bytes(r) == before
    else:
        assert all(is_infinity(g) for g in r[:batch])
        assert bytes(r)[C.sizeof(pb.lib.SecpGej) * batch:] == before[C.sizeof(pb.lib.SecpGej) * batch:]


@pytest.mark.parametrize("handle,first,n,want", [("none", 0, 4, 0), ("none", 0, 0, 1), ("stand_in", 126, 3, 0),
                                                 ("stand_in", 200, 0, 1), ("bn254", 0, 4, 0)])
def test_single_commitment_writes_infinity_before_checking(handle, first, n, want):
    """porla_secp256k1_ecmult_multi_table keeps its contract: r is infinity first, whatever the call returns."""
    t = {"none": None, "stand_in": stand_in(128), "bn254": stand_in(128, pb.CURVE_BN254)}[handle]
    sc, r = garbage(pb.lib.SecpScalar, 4, n), garbage(pb.lib.SecpGej, 1, first)
    assert pb.load().porla_secp256k1_ecmult_multi_table(C.byref(t) if t is not None else None, first, sc, n, r) == want
    assert is_infinity(r[0])
