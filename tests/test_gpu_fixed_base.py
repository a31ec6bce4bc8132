"""Fixed-base scalar multiplication over a one-base look-up table (k_fixed_base_mul, porla_b200/csrc/small_kernels.cuh)
and the client's batched KZG symbols built on it, compute_digest_batch and compute_digest_complement_batch.

  porla_scalar_mul_batch_device : a length-1 table with a look-up table takes k_fixed_base_mul, any other table the
                                  double-and-add of k_scalar_mul; both must give the same bytes and equal the oracle
  compute_digest_batch          : byte-identical to the per-call compute_digest and to [alpha f(tau) mod r]G1
  compute_digest_complement_batch : byte-identical to the per-call compute_digest_complement, following every init_SRS
"""
import ctypes as C
import os
import random
import subprocess
import sys
import threading

import pytest

import porla_b200 as pb
from oracle import curves_py as O

pytestmark = pytest.mark.gpu

BN, SE = O.BN254, O.SECP256K1
CURVES = {"bn254": (pb.CURVE_BN254, BN), "secp256k1": (pb.CURVE_SECP256K1, SE)}
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def enc_point(P, fmt=pb.POINT_BE64):
    if P is None:
        return bytes(64)
    order = "big" if fmt == pb.POINT_BE64 else "little"
    return P[0].to_bytes(32, order) + P[1].to_bytes(32, order)


def enc_scalars(ks, fmt):
    order = "big" if fmt == pb.SCALAR_BE32 else "little"
    return b"".join(k.to_bytes(32, order) for k in ks)


def special_scalars(c):
    """0, 1, order - 1, order, order + 1, multiples of the order, 2^256 - 1, and the n/2 boundary of the secp256k1 recoding."""
    vals = [0, 1, c.n - 1, c.n, c.n + 1, 2 * c.n, 5 * c.n, (1 << 256) - 1, (c.n - 1) // 2, (c.n + 1) // 2, 1 << 254,
            (1 << 255) - 1]
    return [v for v in vals if v < 1 << 256]


def scalar_mul_batch(tab, scalars: bytes, n: int, scalar_fmt: int, out_fmt: int) -> bytes:
    import torch
    lib = pb.load()
    d_sc = torch.frombuffer(bytearray(scalars), dtype=torch.uint8).cuda()
    d_out = torch.full((64 * n,), 0xAB, dtype=torch.uint8, device="cuda")   # every byte must be written
    torch.cuda.synchronize()
    lib.porla_scalar_mul_batch_device(C.c_void_p(tab.handle), C.c_void_p(d_sc.data_ptr()), n, scalar_fmt, out_fmt,
                                      C.c_void_p(d_out.data_ptr()), None)
    torch.cuda.synchronize()
    return d_out.cpu().numpy().tobytes()


def base_point(c, kind, rnd):
    if kind == "G":
        return (c.gx, c.gy)
    if kind == "random":
        return O.mul(c, rnd.randrange(1, c.n), (c.gx, c.gy))
    return None


@pytest.fixture(scope="module")
def lib():
    lib = pb.load()
    lib.porla_device_init()
    return lib


# ------------------------------------------------------------------------------------------- porla_scalar_mul_batch_device
@pytest.mark.parametrize("n,scalar_fmt,out_fmt", [
    (1, pb.SCALAR_BE32, pb.POINT_BE64),
    (129, pb.SCALAR_BE32, pb.POINT_BE64), (129, pb.SCALAR_BE32, pb.POINT_LE64),
    (129, pb.SCALAR_LE32, pb.POINT_BE64), (129, pb.SCALAR_LE32, pb.POINT_LE64),
    ((1 << 16) + 3, pb.SCALAR_BE32, pb.POINT_LE64), ((1 << 16) + 3, pb.SCALAR_LE32, pb.POINT_BE64),
])
@pytest.mark.parametrize("base", ["G", "random", "inf"])
@pytest.mark.parametrize("curve", sorted(CURVES))
def test_fixed_base_table_matches_double_and_add_and_oracle(lib, curve, base, n, scalar_fmt, out_fmt):
    cid, c = CURVES[curve]
    rnd = random.Random(f"{curve}-{base}-{n}-{scalar_fmt}-{out_fmt}")
    B = base_point(c, base, rnd)
    ks = special_scalars(c)[:n] + [rnd.randrange(1 << 256) for _ in range(max(0, n - len(special_scalars(c))))]
    sc = enc_scalars(ks, scalar_fmt)
    plain = pb.Table.from_host(cid, enc_point(B))
    lut = pb.Table.from_host(cid, enc_point(B))
    assert lut.precompute(0, 1, 1) == 8
    try:
        l0 = lib.porla_launch_count()
        got = scalar_mul_batch(lut, sc, n, scalar_fmt, out_fmt)
        assert lib.porla_launch_count() - l0 == 1, "the look-up table path is one launch of k_fixed_base_mul"
        ref = scalar_mul_batch(plain, sc, n, scalar_fmt, out_fmt)
        assert got == ref
        idx = range(n) if n <= 200 else sorted(set(range(len(special_scalars(c)))) | set(rnd.sample(range(n), 48)) | {n - 1})
        for i in idx:
            want = enc_point(None if B is None else O.mul(c, ks[i] % c.n, B), out_fmt)
            assert got[64 * i:64 * i + 64] == want, (i, ks[i])
    finally:
        plain.destroy()
        lut.destroy()


@pytest.mark.parametrize("curve", sorted(CURVES))
def test_wide_window_table(lib, curve):
    """A batch hint of 2^22 gives the one base the c = 16 look-up table (16 windows of 32768 multiples)."""
    cid, c = CURVES[curve]
    rnd = random.Random(77)
    B = base_point(c, "random", rnd)
    n = 4099
    ks = special_scalars(c) + [rnd.randrange(1 << 256) for _ in range(n - len(special_scalars(c)))]
    sc = enc_scalars(ks, pb.SCALAR_BE32)
    plain, lut = pb.Table.from_host(cid, enc_point(B)), pb.Table.from_host(cid, enc_point(B))
    assert lut.precompute(0, 1, 1 << 22) == 16
    try:
        got = scalar_mul_batch(lut, sc, n, pb.SCALAR_BE32, pb.POINT_BE64)
        assert got == scalar_mul_batch(plain, sc, n, pb.SCALAR_BE32, pb.POINT_BE64)
        for i in list(range(len(special_scalars(c)))) + rnd.sample(range(n), 32):
            assert got[64 * i:64 * i + 64] == enc_point(O.mul(c, ks[i] % c.n, B)), i
    finally:
        plain.destroy()
        lut.destroy()


@pytest.mark.parametrize("curve", sorted(CURVES))
def test_million_scalars_checked_by_a_random_combination(lib, curve):
    """2^20 products checked in full without 2^20 oracle multiplications: sum rho_i out_i (an MSM on the device) must be
    [sum rho_i k_i mod order] B for random rho_i; a sample of entries is also checked one by one."""
    cid, c = CURVES[curve]
    n = 1 << 20
    rnd = random.Random(2020 + cid)
    B = base_point(c, "random", rnd)
    raw = rnd.randbytes(32 * n)
    ks = [int.from_bytes(raw[32 * i:32 * i + 32], "big") for i in range(n)]
    lut = pb.Table.from_host(cid, enc_point(B))
    lut.precompute(0, 1, 1)
    try:
        out = scalar_mul_batch(lut, raw, n, pb.SCALAR_BE32, pb.POINT_BE64)
    finally:
        lut.destroy()
    rho_raw = rnd.randbytes(32 * n)
    if cid == pb.CURVE_BN254:
        combo = pb.bn254_multi_exp(out, rho_raw, n)
    else:
        combo = pb.msm_host(cid, rho_raw, out, n)
    total = sum(int.from_bytes(rho_raw[32 * i:32 * i + 32], "big") * ks[i] for i in range(n)) % c.n
    assert combo == enc_point(O.mul(c, total, B))
    for i in rnd.sample(range(n), 24) + [0, n - 1]:
        assert out[64 * i:64 * i + 64] == enc_point(O.mul(c, ks[i] % c.n, B)), i


# ------------------------------------------------------------------------------------------- the client's batched symbols
TAU_KEY = bytes.fromhex("0123456789abcdef0123456789abcdef")
ALPHA_KEY = bytes.fromhex("fedcba9876543210fedcba9876543210")
R = BN.n


def be(x):
    return x.to_bytes(32, "big")


def digest_records(n, batch, tau, rnd):
    """`batch` coefficient records: special records first (all zero; f = (X - tau) g, whose digest is infinity; coefficients
    r, r - 1, r + 1 and 2^256 - 1), then uniform 256-bit coefficients, many of them >= r and >= 2^254."""
    recs = []
    g = [rnd.randrange(R) for _ in range(n - 1)]
    root = [(-tau * g[0]) % R] + [(g[i - 1] - tau * g[i]) % R for i in range(1, n - 1)] + [g[n - 2]]
    edge = [[R, R - 1, R + 1, (1 << 256) - 1][i % 4] for i in range(n)]
    for rec in ([0] * n, root, edge):
        if len(recs) < batch:
            recs.append(rec)
    while len(recs) < batch:
        recs.append([rnd.randrange(1 << 256) for _ in range(n)])
    return recs


@pytest.mark.parametrize("batch", [1, 2, 127, 1024])
def test_digest_batch_matches_per_call_and_oracle(lib, batch):
    n = 200
    tau, alpha = O.fr_set_bytes(TAU_KEY), O.fr_set_bytes(ALPHA_KEY)
    k = pb.Kzg(TAU_KEY, ALPHA_KEY)
    k.init_srs(n)
    rnd = random.Random(batch)
    recs = digest_records(n, batch, tau, rnd)
    data = b"".join(be(v) for rec in recs for v in rec)
    got = k.compute_digest_batch(data, batch)
    assert len(got) == 64 * batch
    G = (BN.gx, BN.gy)
    for j, rec in enumerate(recs):
        assert got[64 * j:64 * j + 64] == k.compute_digest(b"".join(be(v) for v in rec)), j
        if batch <= 127 or j % 16 == 0 or j < 3:
            v = alpha * sum(f * pow(tau, i, R) for i, f in enumerate(rec)) % R
            assert got[64 * j:64 * j + 64] == enc_point(O.mul(BN, v, G)), j
    if batch >= 2:
        assert got[64:128] == bytes(64), "f = (X - tau) g must give the point at infinity"


def test_digest_batch_follows_new_keys_and_srs(lib):
    """The powers alpha tau^i and the base table are rebuilt when init_key / init_SRS change tau, alpha or n_samples."""
    rnd = random.Random(5)
    for tau_key, alpha_key, n in ((TAU_KEY, ALPHA_KEY, 64), (bytes(range(16)), bytes(range(16, 32)), 64),
                                  (bytes(range(16)), bytes(range(16, 32)), 130)):
        k = pb.Kzg(tau_key, alpha_key)
        k.init_srs(n)
        recs = [[rnd.randrange(1 << 256) for _ in range(n)] for _ in range(5)]
        got = k.compute_digest_batch(b"".join(be(v) for rec in recs for v in rec), 5)
        for j, rec in enumerate(recs):
            assert got[64 * j:64 * j + 64] == k.compute_digest(b"".join(be(v) for v in rec)), (n, j)


def complement_scalars(rnd, count):
    return [0, 1, R - 1, R, R + 1, (1 << 256) - 1] + [rnd.randrange(1 << 256) for _ in range(count)]


def test_complement_batch_matches_per_call_and_follows_each_init_srs(lib):
    k = pb.Kzg(TAU_KEY, ALPHA_KEY)
    rnd = random.Random(9)
    ss = complement_scalars(rnd, 200)
    data = b"".join(be(s) for s in ss)
    previous = None
    for _ in range(2):   # the second init_SRS draws a new h_MAC: a stale resident table would still give the old products
        k.init_srs(32)
        H = O.bn254_unmarshal(k.compute_digest_complement(be(1)))
        got = k.compute_digest_complement_batch(data, len(ss))
        for j, s in enumerate(ss):
            assert got[64 * j:64 * j + 64] == k.compute_digest_complement(be(s)), j
            assert got[64 * j:64 * j + 64] == enc_point(O.mul(BN, s % R, H)), j
        assert got != previous
        previous = got
        for b in (1, 3, 4, 5):   # small batches take the leased staging slots
            assert k.compute_digest_complement_batch(data[:32 * b], b) == got[:64 * b]


def test_complement_batch_without_lut_uses_double_and_add(lib, monkeypatch):
    k = pb.Kzg(TAU_KEY, ALPHA_KEY)
    ss = complement_scalars(random.Random(3), 40)
    data = b"".join(be(s) for s in ss)
    monkeypatch.setenv("PORLA_NO_LUT", "1")
    k.init_srs(16)   # the h_MAC table is rebuilt on the next call, now without a look-up table
    k.compute_digest_complement_batch(data, len(ss))
    l0 = lib.porla_launch_count()
    got = k.compute_digest_complement_batch(data, len(ss))
    assert lib.porla_launch_count() - l0 == 2, "k_scalar_mul + export"
    for j, s in enumerate(ss):
        assert got[64 * j:64 * j + 64] == k.compute_digest_complement(be(s)), j
    monkeypatch.delenv("PORLA_NO_LUT")
    k.init_srs(16)


def test_complement_batch_from_eight_threads(lib):
    """Porla's client calls from a pool of 8 threads: concurrent batches of different sizes on different inputs."""
    k = pb.Kzg(TAU_KEY, ALPHA_KEY)
    k.init_srs(16)
    rnd = random.Random(8)
    sizes = [1, 2, 3, 4, 5, 64, 300, 1000]
    inputs = [[rnd.randrange(1 << 256) for _ in range(sizes[t])] for t in range(8)]
    results = [[None] * 6 for _ in range(8)]
    errors = []

    def worker(t):
        try:
            data = b"".join(be(s) for s in inputs[t])
            for r in range(6):
                results[t][r] = k.compute_digest_complement_batch(data, len(inputs[t]))
        except Exception as e:  # pragma: no cover - reported below
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(8)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors
    for t in range(8):
        want = b"".join(k.compute_digest_complement(be(s)) for s in inputs[t])
        for r in range(6):
            assert results[t][r] == want, (t, r)


def test_complement_batch_before_init_srs_is_infinity():
    """Before any init_SRS, h_MAC is the point at infinity: 64 zero bytes per record, as the per-call form gives.  A fresh
    process, since every other test has already drawn an h_MAC."""
    code = (
        "import porla_b200 as pb\n"
        "k = pb.Kzg(bytes(16), bytes(16))\n"
        "data = b''.join((3 * i + 1).to_bytes(32, 'big') for i in range(9))\n"
        "got = k.compute_digest_complement_batch(data, 9)\n"
        "assert got == bytes(64 * 9), got.hex()\n"
        "assert got[:64] == k.compute_digest_complement(data[:32])\n"
        "assert k.compute_digest_complement_batch(b'', 0) == b''\n"
        "print('ok')\n")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]
