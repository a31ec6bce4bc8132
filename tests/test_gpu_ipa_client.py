"""The client side of IPA mode on the B200: MAC complements (porla_secp256k1_ecmult_const_batch) and per-block
commitments (porla_secp256k1_ecmult_multi_table_batch) over resident secp256k1 tables.  Results are checked against the
big-int oracle, and byte for byte against the single-call porla_secp256k1_ecmult_multi_table on the same inputs."""
import ctypes as C
import random
import threading

import pytest

import porla_b200 as pb
from oracle import curves_py as O
from tests.test_ipa_client import TableHead, is_infinity
from tests.test_secp_butterfly import SE, G

pytestmark = pytest.mark.gpu

N = SE.n
EDGES = [0, 1, (N - 1) // 2, (N + 1) // 2, N - 1, N, N + 1, (1 << 256) - 1]   # (n +- 1) / 2: the sign-flip edge


def single(tab, first, scalars):
    """Raw bytes of one porla_secp256k1_ecmult_multi_table call."""
    r = pb.lib.SecpGej()
    assert pb.load().porla_secp256k1_ecmult_multi_table(C.c_void_p(tab.handle), first, pb.lib._scalar_array(scalars),
                                                        len(scalars), C.byref(r)) == 1
    return bytes(r)


def const_batch_raw(base, scalars):
    r = (pb.lib.SecpGej * max(1, len(scalars)))()
    ok = pb.load().porla_secp256k1_ecmult_const_batch(C.c_void_p(base.handle), pb.lib._scalar_array(scalars), len(scalars), r)
    return ok, r


def multi_batch_raw(tab, first, scalars, n, batch):
    r = (pb.lib.SecpGej * max(1, batch))()
    ok = pb.load().porla_secp256k1_ecmult_multi_table_batch(C.c_void_p(tab.handle), first, pb.lib._scalar_array(scalars), n,
                                                            batch, r)
    return ok, r


_TABLES = {}


def table(name):
    """(points, resident table): h alone, infinity alone, 1025 generators, and 128 generators followed by h."""
    if name not in _TABLES:
        rnd = random.Random(name)
        h = O.mul(SE, rnd.randrange(1, N), G)
        pts = {"h": [h], "inf": [None], "gens1025": [O.mul(SE, rnd.randrange(1, N), G) for _ in range(1025)]}.get(name)
        if name == "gens_h129":
            pts = table("gens1025")[0][:128] + table("h")[0]
        _TABLES[name] = (pts, pb.SecpGenerators(pts))
    return _TABLES[name]


def test_stand_in_layout_of_the_cpu_tests_matches_a_real_table():
    for name, length in (("h", 1), ("gens_h129", 129)):
        head = TableHead.from_address(table(name)[1].handle)
        assert (head.n, head.curve) == (length, pb.CURVE_SECP256K1)
    bn = pb.Table.multiples_of_generator(pb.CURVE_BN254, (5).to_bytes(32, "little") * 3, 3)
    head = TableHead.from_address(bn.handle)
    assert (head.n, head.curve) == (3, pb.CURVE_BN254)
    bn.destroy()


# ---------------------------------------------------------------------------- MAC complements
@pytest.mark.parametrize("batch", [1, 4, 5, 1000, 4096])
def test_complements_against_oracle_and_single_calls(batch):
    (h,), base = table("h")
    rnd = random.Random(batch)
    k = batch % len(EDGES)
    pool = EDGES[k:] + EDGES[:k] if batch < len(EDGES) else EDGES
    scalars = (pool + [rnd.randrange(1 << 256) for _ in range(batch)])[:batch]
    ok, got = pb.secp256k1_ecmult_const_batch(base, scalars)
    assert ok == 1 and len(got) == batch
    checked = range(batch) if batch <= 1000 else sorted(set(range(len(EDGES))) | set(rnd.sample(range(batch), 300)))
    for i in checked:
        s = scalars[i] % N
        assert got[i] == (O.mul(SE, s, h) if s else None), (i, hex(scalars[i]))
    ok, raw = const_batch_raw(base, scalars)
    assert ok == 1
    for i in range(batch):
        assert bytes(raw[i]) == single(base, 0, [scalars[i]]), i
    for i in range(min(batch, len(EDGES))):
        if scalars[i] % N == 0:
            assert is_infinity(raw[i])


def test_complements_of_an_infinite_base_are_infinity():
    _, base = table("inf")
    scalars = EDGES + [random.Random(3).randrange(1 << 256) for _ in range(9)]
    ok, raw = const_batch_raw(base, scalars)
    assert ok == 1
    assert all(is_infinity(g) for g in raw[:len(scalars)])


# ---------------------------------------------------------------------------- per-block commitments
def blocks(n, batch, seed):
    rnd = random.Random(seed)
    sc = [rnd.randrange(1 << 256) for _ in range(n * batch)]
    sc[:min(len(sc), len(EDGES))] = EDGES[:len(sc)]
    if batch > 1:                                   # block 1 of all-zero scalars: infinity
        sc[n:2 * n] = [0] * n
    return sc


def check_blocks(tab_name, first, n, batch, scalars, got, raw, full):
    """Every block against the oracle's multi-exponentiation (all blocks up to `full`, then a sample) and bytewise
    against its single call."""
    pts = table(tab_name)[0][first:first + n]
    rnd = random.Random(n * batch)
    checked = range(batch) if batch <= full else sorted({0, 1, batch - 1} | set(rnd.sample(range(batch), full)))
    tab = table(tab_name)[1]
    for b in checked:
        blk = scalars[b * n:(b + 1) * n]
        assert got[b] == O.msm(SE, [s % N for s in blk], pts), b
    for b in range(batch):
        assert bytes(raw[b]) == single(tab, first, scalars[b * n:(b + 1) * n]), b


@pytest.mark.parametrize("first,n,batch,full", [(0, 128, 1, 1), (0, 128, 4, 4), (0, 128, 5, 5), (0, 128, 1024, 4),
                                                (1, 127, 6, 6), (0, 1024, 4, 1), (0, 1025, 4, 1)])
def test_commitments_against_oracle_and_single_calls(first, n, batch, full):
    """4 x 1024 terms lease a staging slot, 4 x 1025 take the shared staging area; 5 blocks pass the slot's batch limit."""
    tab_name = "gens1025" if n > 128 else "gens_h129"
    tab = table(tab_name)[1]
    scalars = blocks(n, batch, 7 * n + batch + first)
    ok, got = tab.multi_batch(first, scalars, n, batch)
    assert ok == 1 and len(got) == batch
    ok, raw = multi_batch_raw(tab, first, scalars, n, batch)
    assert ok == 1
    check_blocks(tab_name, first, n, batch, scalars, got, raw, full)
    if batch > 1:
        assert got[1] is None and is_infinity(raw[1])


def test_whole_mac_as_one_129_term_block():
    """h appended to the generator table, the PRF value after the chunks: commitment plus complement in one block."""
    pts, tab = table("gens_h129")
    gens, h = pts[:128], pts[128]
    rnd = random.Random(129)
    batch = 8
    chunks = [[rnd.randrange(1 << 256) for _ in range(128)] for _ in range(batch)]
    prf = [rnd.randrange(1 << 256) for _ in range(batch)]
    prf[1], prf[2] = 0, N
    scalars = [s for b in range(batch) for s in chunks[b] + [prf[b]]]
    ok, got = tab.multi_batch(0, scalars, 129, batch)
    assert ok == 1
    for b in range(3):
        assert got[b] == O.add(SE, O.msm(SE, [s % N for s in chunks[b]], gens), O.mul(SE, prf[b] % N, h)), b
    ok, raw = multi_batch_raw(tab, 0, scalars, 129, batch)
    assert ok == 1
    (hh,), base = table("h")
    for b in range(batch):
        assert bytes(raw[b]) == single(tab, 0, scalars[b * 129:(b + 1) * 129]), b
        # the same MAC from the two separate entries: the commitment, then the complement, added
        ok, comp = pb.secp256k1_ecmult_const_batch(base, [prf[b]])
        assert hh == h and ok == 1
        assert got[b] == O.add(SE, tab.multi(0, chunks[b])[1], comp[0]), b


# ---------------------------------------------------------------------------- refused shapes on real tables
def test_refused_shapes_on_real_tables_leave_buffers_untouched():
    lib = pb.load()
    _, gens = table("gens_h129")
    bn = pb.Table.multiples_of_generator(pb.CURVE_BN254, (5).to_bytes(32, "little"), 1)
    rnd = random.Random(11)
    sc = (pb.lib.SecpScalar * 256).from_buffer_copy(rnd.randbytes(32 * 256))
    for handle, n in ((gens.handle, 1), (gens.handle, 4), (bn.handle, 4)):          # length 129, a BN254 base
        r = (pb.lib.SecpGej * 4)()
        C.memset(r, 0x5A, C.sizeof(r))
        assert lib.porla_secp256k1_ecmult_const_batch(C.c_void_p(handle), sc, n, r) == 0
        assert bytes(r) == b"\x5a" * C.sizeof(r)
    for handle, first, n, batch in ((gens.handle, 0, 130, 1), (gens.handle, 2, 128, 1), (gens.handle, 129, 1, 2),
                                    (gens.handle, 0, 128, 1 << 24), (gens.handle, 0, 1, 1 << 31), (bn.handle, 0, 1, 1)):
        r = (pb.lib.SecpGej * 4)()
        C.memset(r, 0x5A, C.sizeof(r))
        before = bytes(sc)
        assert lib.porla_secp256k1_ecmult_multi_table_batch(C.c_void_p(handle), first, sc, n, batch, r) == 0, (first, n, batch)
        assert bytes(r) == b"\x5a" * C.sizeof(r) and bytes(sc) == before
    assert gens.multi_batch(2, [1] * 128, 128, 1) == (0, None)
    bn.destroy()


# ---------------------------------------------------------------------------- concurrency
def test_concurrent_complements_and_commitments_equal_their_serial_values():
    """Porla's pool threads issue per-block commitments and complements at once.  Eight threads, each with its own
    scalars, several rounds: small calls lease staging slots, the larger complement batches of odd threads take the shared
    staging area alongside them.  Every result equals the serial one."""
    _, base = table("h")
    _, gens = table("gens_h129")
    T, rounds = 8, 4
    rnd = random.Random(88)
    comp = [[rnd.randrange(1 << 256) for _ in range(3 if t % 2 == 0 else 64)] for t in range(T)]
    com = [[rnd.randrange(1 << 256) for _ in range(2 * 129)] for _ in range(T)]
    want_comp = [bytes(const_batch_raw(base, comp[t])[1]) for t in range(T)]
    want_com = [bytes(multi_batch_raw(gens, 0, com[t], 129, 2)[1]) for t in range(T)]
    errors = []

    def worker(t):
        for _ in range(rounds):
            ok, r = const_batch_raw(base, comp[t])
            if ok != 1 or bytes(r) != want_comp[t]:
                errors.append(("complement", t))
            ok, r = multi_batch_raw(gens, 0, com[t], 129, 2)
            if ok != 1 or bytes(r) != want_com[t]:
                errors.append(("commitment", t))

    th = [threading.Thread(target=worker, args=(t,)) for t in range(T)]
    [x.start() for x in th]
    [x.join() for x in th]
    assert not errors, errors[:6]
    assert want_comp[0] != want_comp[2] and want_com[0] != want_com[1]
