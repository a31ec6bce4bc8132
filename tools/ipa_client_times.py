"""Wall-clock times of the IPA-mode client entries on one GPU, against the per-call routes the library offered before them.

    python tools/ipa_client_times.py [--out FILE]

  complements   porla_secp256k1_ecmult_const_batch at batch 1 / 2 / 4 / 8 / 16 / 128 / 1024 / 4096 over a length-1 table
                of h, scalars in pageable (ctypes array) and pinned (torch pin_memory) caller buffers, against one
                porla_secp256k1_ecmult_multi_table(base, 0, &k, 1) call per scalar; the KZG twin
                compute_digest_complement_batch (pageable) is timed alongside for reference
  commitments   porla_secp256k1_ecmult_multi_table_batch over 1 / 16 / 128 / 1024 blocks of 128 chunks, pageable and
                pinned scalars, against one porla_secp256k1_ecmult_multi_table call per block; then the whole MAC as one
                block of 129 terms (generators followed by h, the chunks followed by the PRF value)
Every entry returns its results to the host and ends in a device synchronise, so a wall clock around the call covers
the device work.  Median of 7 calls after one warm-up call of the same shape; before timing, each pair of routes is
checked to give identical bytes.  The card's name and power limit are read first, in the same run.  libsecp256k1's own
secp256k1_ecmult_const (the reference's host route) is not built here, so that comparison is not measured.
"""
import argparse
import ctypes as C
import os
import random
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

REPS = 7


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def timed(fn):
    """Median wall time in ms of fn() over REPS calls after one warm-up."""
    ws = []
    for i in range(REPS + 1):
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

    import torch

    import porla_b200 as pb
    from oracle import curves_py as O
    from porla_b200.lib import _slice
    lib = pb.load()
    lib.porla_device_init()
    SE = O.SECP256K1
    G = (SE.gx, SE.gy)
    rnd = random.Random(6)
    chunks = 128
    h = O.mul(SE, rnd.randrange(1, SE.n), G)
    gens_pts = [O.mul(SE, rnd.randrange(1, SE.n), G) for _ in range(chunks)]
    base = pb.SecpGenerators([h])
    gens = pb.SecpGenerators(gens_pts + [h])
    Gej, Sc = pb.lib.SecpGej, pb.lib.SecpScalar

    def scalars(count, pinned):
        """A secp256k1_scalar array of `count` random values: a ctypes array (pageable) or a view of pinned memory."""
        raw = rnd.randbytes(32 * count)
        if not pinned:
            return (Sc * count).from_buffer_copy(raw), None
        t = torch.empty(32 * count, dtype=torch.uint8, pin_memory=True)
        t[:] = torch.frombuffer(bytearray(raw), dtype=torch.uint8)
        return (Sc * count).from_address(t.data_ptr()), t

    emit("MAC complements: porla_secp256k1_ecmult_const_batch pageable / pinned | one ecmult_multi_table(base, 0, &k, 1) "
         "per scalar | KZG twin compute_digest_complement_batch (pageable); libsecp256k1 ecmult_const: not measured")
    kzg = pb.Kzg(bytes.fromhex("ffeeddccbbaa99887766554433221100"), bytes.fromhex("00112233445566778899aabbccddeeff"))
    kzg.init_srs(chunks)
    for batch in (1, 2, 4, 8, 16, 128, 1024, 4096):
        r = (Gej * batch)()
        t_new = {}
        for kind in ("pageable", "pinned"):
            sc, keep = scalars(batch, kind == "pinned")
            assert lib.porla_secp256k1_ecmult_const_batch(C.c_void_p(base.handle), sc, batch, r) == 1
            one = Gej()
            for i in range(0, batch, max(1, batch // 16)):
                assert lib.porla_secp256k1_ecmult_multi_table(C.c_void_p(base.handle), 0, C.byref(sc[i]), 1, C.byref(one)) == 1
                assert bytes(one) == bytes(r[i]), ("batched complement differs from the single call", batch, i)
            t_new[kind] = timed(lambda: lib.porla_secp256k1_ecmult_const_batch(C.c_void_p(base.handle), sc, batch, r))
        one = Gej()

        def per_scalar():
            for i in range(batch):
                lib.porla_secp256k1_ecmult_multi_table(C.c_void_p(base.handle), 0, C.byref(sc[i]), 1, C.byref(one))

        t_old = timed(per_scalar)
        kin, kout = _slice(bytearray(rnd.randbytes(32 * batch))), _slice(bytearray(64 * batch))
        t_kzg = timed(lambda: lib.compute_digest_complement_batch(C.byref(kin), batch, C.byref(kout)))
        emit("  %5d scalars  %8.3f / %8.3f ms | %9.3f ms  (%5.1fx) | KZG twin %8.3f ms"
             % (batch, t_new["pageable"], t_new["pinned"], t_old, t_old / t_new["pageable"], t_kzg))

    emit("per-block commitments, %d chunks: porla_secp256k1_ecmult_multi_table_batch pageable / pinned | one "
         "ecmult_multi_table call per block" % chunks)
    for n, label in ((chunks, "commitment"), (chunks + 1, "whole MAC, 129 terms")):
        if n != chunks:
            emit("%s: the same entry over the generators followed by h" % label)
        for batch in (1, 16, 128, 1024):
            r = (Gej * batch)()
            t_new = {}
            for kind in ("pageable", "pinned"):
                sc, keep = scalars(n * batch, kind == "pinned")
                assert lib.porla_secp256k1_ecmult_multi_table_batch(C.c_void_p(gens.handle), 0, sc, n, batch, r) == 1
                one = Gej()
                for b in range(0, batch, max(1, batch // 16)):
                    assert lib.porla_secp256k1_ecmult_multi_table(C.c_void_p(gens.handle), 0, C.byref(sc[n * b]), n,
                                                                  C.byref(one)) == 1
                    assert bytes(one) == bytes(r[b]), ("batched block differs from the single call", n, batch, b)
                t_new[kind] = timed(lambda: lib.porla_secp256k1_ecmult_multi_table_batch(C.c_void_p(gens.handle), 0, sc, n,
                                                                                         batch, r))
            one = Gej()

            def per_block():
                for b in range(batch):
                    lib.porla_secp256k1_ecmult_multi_table(C.c_void_p(gens.handle), 0, C.byref(sc[n * b]), n, C.byref(one))

            t_old = timed(per_block)
            emit("  %5d blocks   %8.3f / %8.3f ms | %9.3f ms  (%5.1fx)"
                 % (batch, t_new["pageable"], t_new["pinned"], t_old, t_old / t_new["pageable"]))
    base.destroy()
    gens.destroy()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
