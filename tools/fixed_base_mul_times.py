"""Times of the fixed-base scalar multiplications: the client's per-call KZG symbols against their batched forms, and
porla_scalar_mul_batch_device on a length-1 table without a look-up table (double-and-add, k_scalar_mul) and with one
(k_fixed_base_mul).  Every pair of paths it compares is first checked to produce identical bytes.  Prints one JSON line
with the card's name and power limit, read in the same run.

    python tools/fixed_base_mul_times.py [--n-samples 128] [--batches 1,2,4,8,16,128,1024,4096] [--lgs 16,20,24]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import porla_b200 as pb
from porla_b200.lib import _ptr_slice, _slice


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True)
    if q.returncode != 0:
        return {"name": torch.cuda.get_device_name(0), "power_limit_w": None, "max_sm_clock_mhz": None}
    name, pl, clk = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit_w": float(pl), "max_sm_clock_mhz": float(clk)}


def wall_ms(fn, min_s=0.3, max_reps=200, warmup=2):
    """Median wall time of fn() in ms; every call under test ends in a device synchronise."""
    for _ in range(warmup):
        fn()
    ts, t_end = [], time.perf_counter() + min_s
    while len(ts) < 3 or (time.perf_counter() < t_end and len(ts) < max_reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


class Buf:
    """A host buffer the symbols read or write through a GoSlice: pageable (bytearray) or page-locked (torch pinned)."""

    def __init__(self, data, pinned):
        self.n = len(data)
        if pinned:
            self.t = torch.empty(max(1, self.n), dtype=torch.uint8, pin_memory=True)
            if self.n:
                self.t[:self.n] = torch.frombuffer(bytearray(data), dtype=torch.uint8)
            self.slice = _ptr_slice(self.t.data_ptr(), self.n)
        else:
            self.b = bytearray(data)
            self.slice = _slice(self.b)

    def bytes(self):
        return self.t[:self.n].numpy().tobytes() if hasattr(self, "t") else bytes(self.b)


def host_symbols(lib, k, n_samples, batches):
    g = torch.Generator().manual_seed(7)
    bmax = max(batches)
    coeffs = torch.randint(0, 256, (bmax * n_samples * 32,), dtype=torch.uint8, generator=g).numpy().tobytes()
    scalars = torch.randint(0, 256, (bmax * 32,), dtype=torch.uint8, generator=g).numpy().tobytes()
    # per-call reference bytes (also what the per-call timing runs)
    rec = n_samples * 32
    want_d = b"".join(k.compute_digest(coeffs[rec * j:rec * (j + 1)]) for j in range(bmax))
    want_c = b"".join(k.compute_digest_complement(scalars[32 * j:32 * (j + 1)]) for j in range(bmax))
    rows = []
    for b in batches:
        row = {"batch": b}
        ins_d = [bytearray(coeffs[rec * j:rec * (j + 1)]) for j in range(b)]
        ins_c = [bytearray(scalars[32 * j:32 * (j + 1)]) for j in range(b)]
        outs = [bytearray(64) for _ in range(b)]
        sl_d = [(_slice(x), _slice(o)) for x, o in zip(ins_d, outs)]
        sl_c = [(_slice(x), _slice(o)) for x, o in zip(ins_c, outs)]

        def per_call(fn, sl):
            def run():
                for a, o in sl:
                    fn(C.byref(a), C.byref(o))
            return run

        row["per_call_digest_ms"] = wall_ms(per_call(lib.compute_digest, sl_d), warmup=1)
        row["per_call_complement_ms"] = wall_ms(per_call(lib.compute_digest_complement, sl_c), warmup=1)
        for kind in ("pageable", "pinned"):
            pinned = kind == "pinned"
            din, dout = Buf(coeffs[:rec * b], pinned), Buf(bytes(64 * b), pinned)
            cin, cout = Buf(scalars[:32 * b], pinned), Buf(bytes(64 * b), pinned)
            fd = lambda: lib.compute_digest_batch(C.byref(din.slice), b, C.byref(dout.slice))
            fc = lambda: lib.compute_digest_complement_batch(C.byref(cin.slice), b, C.byref(cout.slice))
            fd()
            fc()
            assert dout.bytes() == want_d[:64 * b], ("compute_digest_batch differs from compute_digest", b, kind)
            assert cout.bytes() == want_c[:64 * b], ("compute_digest_complement_batch differs from the per-call form", b, kind)
            row["batch_digest_%s_ms" % kind] = wall_ms(fd)
            row["batch_complement_%s_ms" % kind] = wall_ms(fc)
        rows.append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
    return rows


def device_events_ms(fn, reps):
    st = torch.cuda.current_stream()
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        fn()
        e1.record(st)
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return statistics.median(ts)


def device_scalar_mul(lib, lgs):
    rows = []
    st = torch.cuda.current_stream().cuda_stream
    gen = {pb.CURVE_BN254: (1, 2),
           pb.CURVE_SECP256K1: (0x79BE667EF9DCBBAC55A06295CE870B07029BFCDB2DCE28D959F2815B16F81798,
                                0x483ADA7726A3C4655DA4FBFC0E1108A8FD17B448A68554199C47D08FFB10D4B8)}
    for curve, name in ((pb.CURVE_BN254, "bn254"), (pb.CURVE_SECP256K1, "secp256k1")):
        x, y = gen[curve]
        base = x.to_bytes(32, "big") + y.to_bytes(32, "big")
        plain, lut = pb.Table.from_host(curve, base), pb.Table.from_host(curve, base)
        c = lut.precompute(0, 1, 1)
        for lg in lgs:
            n = 1 << lg
            g = torch.Generator(device="cuda").manual_seed(lg)
            sc = torch.randint(-2**31, 2**31 - 1, (n, 8), dtype=torch.int32, device="cuda", generator=g)
            o_plain = torch.empty(64 * n, dtype=torch.uint8, device="cuda")
            o_lut = torch.empty(64 * n, dtype=torch.uint8, device="cuda")
            run = lambda t, o: lib.porla_scalar_mul_batch_device(C.c_void_p(t.handle), C.c_void_p(sc.data_ptr()), n, pb.SCALAR_LE32,
                                                                 pb.POINT_BE64, C.c_void_p(o.data_ptr()), C.c_void_p(st))
            run(plain, o_plain)
            run(lut, o_lut)
            torch.cuda.synchronize()
            assert torch.equal(o_plain, o_lut), ("look-up table path differs from double-and-add", name, lg)
            reps = 5 if lg >= 22 else 20
            t_plain = device_events_ms(lambda: run(plain, o_plain), reps)
            t_lut = device_events_ms(lambda: run(lut, o_lut), reps)
            row = {"curve": name, "scalars": n, "lut_window": c, "double_and_add_ms": t_plain, "lut_ms": t_lut,
                   "speedup": t_plain / t_lut}
            rows.append(row)
            print(json.dumps(row), file=sys.stderr, flush=True)
            del sc, o_plain, o_lut
            torch.cuda.empty_cache()
        plain.destroy()
        lut.destroy()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-samples", type=int, default=128)
    ap.add_argument("--batches", default="1,2,4,8,16,128,1024,4096")
    ap.add_argument("--lgs", default="16,20,24")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: these are GPU timings")
    lib = pb.load()
    lib.porla_device_init()
    info = card()
    k = pb.Kzg(bytes.fromhex("ffeeddccbbaa99887766554433221100"), bytes.fromhex("00112233445566778899aabbccddeeff"))
    k.init_srs(a.n_samples)
    host = host_symbols(lib, k, a.n_samples, [int(x) for x in a.batches.split(",")])
    dev = device_scalar_mul(lib, [int(x) for x in a.lgs.split(",")])
    print(json.dumps({"tool": "fixed_base_mul_times", "card": info, "n_samples": a.n_samples, "host_symbols": host,
                      "scalar_mul_batch_device": dev}))


if __name__ == "__main__":
    main()
