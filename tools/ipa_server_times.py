"""Wall-clock times of the IPA-mode server entries on one GPU, against the per-call routes the library offered before them.

    python tools/ipa_server_times.py [--out FILE]

  align       porla_secp256k1_align_mac_batch on 1 / 16 / 128 / 1024 blocks of 128 chunks (values below LCM_IPA), against
              one porla_secp256k1_ecmult_multi_table call per block on the already reduced scalars c_i (the scalar
              preparation those calls need, 512-bit arithmetic on the host, is not counted for them)
  aggregate   porla_secp256k1_audit_aggregate over 128 / 766 / 4096 blocks of 128 chunks
  gej         porla_secp256k1_ecmult_multi_gej at n = 128 and 766 with nbatch = 2 on Jacobian MACs with random z, against
              the drop-in route on the same points as secp256k1_ge: one host gej -> ge conversion per point (timed through
              porla_secp256k1_gej_serialize, one host field inversion each, ctypes call included) plus two porla_msm_host
              calls, the multi-exponentiation porla_secp256k1_ecmult_multi_var runs after its callbacks
Every entry returns its results to the host, so a wall clock around the call covers the device work.  Median of 7 calls
after one warm-up call of the same shape.  The card's name and power limit are read first, in the same run.
"""
import argparse
import ctypes as C
import os
import random
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

PRIME = 207 * 2**248 + 1
REPS = 7


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def timed(fn, prepare=None):
    """Median wall time in ms of fn() over REPS calls after one warm-up; prepare() runs untimed before each call."""
    ws = []
    for i in range(REPS + 1):
        if prepare:
            prepare()
        t0 = time.perf_counter()
        fn()
        dt = (time.perf_counter() - t0) * 1e3
        if i:
            ws.append(dt)
    return median(ws)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    emit("card: " + (q.stdout.strip().splitlines()[0] if q.stdout.strip() else "unknown"))

    import porla_b200 as pb
    from oracle import curves_py as O
    lib = pb.load()
    lib.porla_device_init()
    SE = O.SECP256K1
    G = (SE.gx, SE.gy)
    LCM = PRIME * SE.n
    rnd = random.Random(5)
    chunks = 128
    gens = pb.SecpGenerators([O.mul(SE, rnd.randrange(1, SE.n), G) for _ in range(chunks)])

    emit("align_MAC, %d chunks per block: porla_secp256k1_align_mac_batch | one ecmult_multi_table call per block" % chunks)
    for batch in (1, 16, 128, 1024):
        vals = [rnd.randrange(LCM) for _ in range(batch * chunks)]
        pristine = b"".join(v.to_bytes(64, "little") for v in vals)
        data = bytearray(pristine)
        out = (pb.lib.SecpGej * batch)()
        dp = pb.lib._as_void_p(data)

        def refill():
            data[:] = pristine

        t_new = timed(lambda: lib.porla_secp256k1_align_mac_batch(C.c_void_p(gens.handle), chunks, dp, batch, out), refill)
        sc = (pb.lib.SecpScalar * (batch * chunks)).from_buffer_copy(
            b"".join((((v % PRIME) - v) % SE.n).to_bytes(32, "little") for v in vals))
        r = pb.lib.SecpGej()
        base = C.addressof(sc)

        def per_block():
            for b in range(batch):
                lib.porla_secp256k1_ecmult_multi_table(C.c_void_p(gens.handle), 0, C.cast(base + 32 * chunks * b,
                                                       C.POINTER(pb.lib.SecpScalar)), chunks, C.byref(r))

        t_old = timed(per_block)
        emit("  %5d blocks   %9.3f ms | %9.3f ms   (%.1fx)" % (batch, t_new, t_old, t_old / t_new))

    emit("audit aggregation + align_MAC on B, %d chunks per block: porla_secp256k1_audit_aggregate" % chunks)
    for n in (128, 766, 4096):
        coefs = b"".join(rnd.randrange(1 << 31).to_bytes(4, "little") for _ in range(n))
        blocks = rnd.randbytes(64 * chunks * n)
        blocks = b"".join((int.from_bytes(blocks[64 * i:64 * i + 64], "little") % LCM).to_bytes(64, "little")
                          for i in range(n * chunks))
        b_out, al = bytearray(32 * chunks), pb.lib.SecpGej()
        cp, bp, op = pb.lib._as_void_p(coefs), pb.lib._as_void_p(blocks), pb.lib._as_void_p(b_out)
        t = timed(lambda: lib.porla_secp256k1_audit_aggregate(C.c_void_p(gens.handle), chunks, cp, bp, n, op, C.byref(al)))
        emit("  %5d blocks   %9.3f ms" % (n, t))

    emit("multi-exponentiation of Jacobian MACs, nbatch = 2: ecmult_multi_gej | gej -> ge on the host + 2 x porla_msm_host"
         " = total")
    for n in (128, 766):
        total = 2 * n
        ks = [rnd.randrange(1, SE.n) for _ in range(total)]
        t = pb.Table.multiples_of_generator(pb.CURVE_SECP256K1, b"".join(k.to_bytes(32, "little") for k in ks), total)
        raw = t.export(pb.POINT_LE64)
        t.destroy()
        gejs = (pb.lib.SecpGej * total)()
        for i in range(total):
            x, y = int.from_bytes(raw[64 * i:64 * i + 32], "little"), int.from_bytes(raw[64 * i + 32:64 * i + 64], "little")
            z = rnd.randrange(2, SE.p)
            gejs[i].x, gejs[i].y = pb.lib._int_to_fe(x * z * z % SE.p), pb.lib._int_to_fe(y * pow(z, 3, SE.p) % SE.p)
            gejs[i].z, gejs[i].infinity = pb.lib._int_to_fe(z), 0
        scal = [rnd.randrange(SE.n) for _ in range(total)]
        sc = (pb.lib.SecpScalar * total).from_buffer_copy(b"".join(s.to_bytes(32, "little") for s in scal))
        r = (pb.lib.SecpGej * 2)()
        t_gej = timed(lambda: lib.porla_secp256k1_ecmult_multi_gej(gejs, sc, n, 2, r))
        ser = (C.c_char * 33)()

        def convert():
            for i in range(total):
                lib.porla_secp256k1_gej_serialize(C.byref(gejs[i]), ser)

        t_conv = timed(convert)
        sb, pts = bytes(sc), raw
        out = (C.c_ubyte * 64)()

        def two_msms():
            for b in range(2):
                lib.porla_msm_host(pb.CURVE_SECP256K1, sb[32 * n * b:32 * n * (b + 1)], pts[64 * n * b:64 * n * (b + 1)], n, 1,
                                   pb.SCALAR_LE32, pb.POINT_LE64, C.cast(out, C.c_void_p))

        t_msm = timed(two_msms)
        old = t_conv + t_msm
        emit("  n = %4d   %9.3f ms | %7.3f + %7.3f = %9.3f ms   (conversion %.0f%% of the old route, %.1fx)"
             % (n, t_gej, t_conv, t_msm, old, 100 * t_conv / old, old / t_gej))
    gens.destroy()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
