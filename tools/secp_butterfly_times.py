"""Per-stage time of the secp256k1 FFT in the exponent (IPA-mode rebuild butterflies) on every route, one B200.

    python tools/secp_butterfly_times.py [--compare NAME=TREE ...]

For 1 ... 131 072 butterflies per stage (a resident table of 2 nb points, m = 2 nb, twiddles on the device):
  quad        k_butterfly_quad, four lanes per butterfly (PORLA_BUTTERFLY_QUAD=1)
  one_thread  k_butterfly, one thread per butterfly, GLV joint double-and-add (PORLA_BUTTERFLY_QUAD=0)
  default     the route butterfly_impl picks
  host        porla_secp256k1_butterfly_stage on the calling host's threads (PORLA_HOST_BUTTERFLIES large; up to 4096)
Device times: CUDA events around 10 back-to-back stages, median of 5 windows.  Host times: wall clock, median of 5.
Each --compare NAME=TREE times the default route of another built tree's porla_b200 package (e.g. an earlier commit, whose
secp256k1 stage is the plain 256-bit double-and-add) in a subprocess.  Then the 10 stages of one 1024-MAC rebuild side through porla_secp256k1_butterfly_stage
with its default routes.  The card's name and power limit are printed first.
"""
import argparse
import ctypes as C
import os
import random
import subprocess
import sys
import time

sys.path.insert(0, os.environ.get("PORLA_TREE") or os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SIZES = [1 << i for i in range(18)]   # 1 ... 131 072: past the 75 776 butterflies (148 SMs x 512) of the compact-type route


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def device_times(routes):
    import torch
    import porla_b200 as pb
    lib = pb.load()
    rnd = random.Random(1)
    n_sc = 2 * SIZES[-1]
    d_tw = torch.frombuffer(bytearray(b"".join(rnd.randrange(1 << 256).to_bytes(32, "big") for _ in range(n_sc // 2))),
                            dtype=torch.uint8).cuda()
    ks = b"".join(rnd.randrange(1, 1 << 255).to_bytes(32, "little") for _ in range(n_sc))
    stream = torch.cuda.current_stream()
    out = {}
    for route in routes:
        if route == "quad":
            os.environ["PORLA_BUTTERFLY_QUAD"] = "1"
        elif route == "one_thread":
            os.environ["PORLA_BUTTERFLY_QUAD"] = "0"
        else:
            os.environ.pop("PORLA_BUTTERFLY_QUAD", None)
        for nb in SIZES:
            n = 2 * nb
            t = pb.Table.multiples_of_generator(pb.CURVE_SECP256K1, ks[:32 * n], n)
            stage = lambda: lib.porla_butterfly_stage_device(C.c_void_p(t.handle), n, C.c_void_p(d_tw.data_ptr()),
                                                             pb.SCALAR_BE32, 1, C.c_void_p(stream.cuda_stream))
            stage()
            torch.cuda.synchronize()
            ws = []
            for _ in range(5):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(10):
                    stage()
                e1.record()
                e1.synchronize()
                ws.append(e0.elapsed_time(e1) / 10)
            out[(route, nb)] = median(ws)
            print("%-10s %6d butterflies  %8.3f ms/stage" % (route, nb, out[(route, nb)]), flush=True)
            t.destroy()
    return out


def gej_array(n, rnd):
    import porla_b200 as pb
    from oracle import curves_py as O
    se = O.SECP256K1
    t = pb.Table.multiples_of_generator(pb.CURVE_SECP256K1, b"".join(rnd.randrange(1, se.n).to_bytes(32, "little")
                                                                        for _ in range(n)), n)
    raw = t.export(pb.POINT_LE64)
    t.destroy()
    arr = (pb.lib.SecpGej * n)()
    for i in range(n):
        x, y = int.from_bytes(raw[64 * i:64 * i + 32], "little"), int.from_bytes(raw[64 * i + 32:64 * i + 64], "little")
        arr[i].x, arr[i].y, arr[i].z, arr[i].infinity = pb.lib._int_to_fe(x), pb.lib._int_to_fe(y), pb.lib._int_to_fe(1), 0
    return arr


def host_times():
    import porla_b200 as pb
    os.environ["PORLA_HOST_BUTTERFLIES"] = str(1 << 30)
    rnd = random.Random(2)
    out = {}
    for nb in [s for s in SIZES if s <= 4096]:
        arr = gej_array(2 * nb, rnd)
        tw = [rnd.randrange(1 << 256) for _ in range(nb)]
        ws = []
        for _ in range(5):
            t0 = time.perf_counter()
            pb.secp256k1_butterfly_stage(arr, 2 * nb, tw)
            ws.append((time.perf_counter() - t0) * 1e3)
        out[("host", nb)] = median(ws)
        print("%-10s %6d butterflies  %8.3f ms/stage" % ("host", nb, out[("host", nb)]), flush=True)
    del os.environ["PORLA_HOST_BUTTERFLIES"]
    return out


def rebuild_side():
    import porla_b200 as pb
    rnd = random.Random(3)
    n = 1024
    arr = gej_array(n, rnd)
    pb.secp256k1_butterfly_stage(gej_array(4, rnd), 2, [5])          # warm-up of the small path
    pb.secp256k1_butterfly_stage(gej_array(512, rnd), 512, [5] * 256)  # and of the device path
    total, m = 0.0, 2
    print("one 1024-MAC rebuild side through porla_secp256k1_butterfly_stage (default routes):")
    while m <= n:
        tw = [rnd.randrange(1 << 256) for _ in range(m // 2)]
        t0 = time.perf_counter()
        assert pb.secp256k1_butterfly_stage(arr, m, tw) == 1
        dt = (time.perf_counter() - t0) * 1e3
        total += dt
        print("  m = %4d (512 butterflies)  %8.3f ms" % (m, dt), flush=True)
        m *= 2
    print("  10 stages                  %8.3f ms" % total, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--compare", action="append", default=[], help="NAME=path/to/built/tree: its default route")
    ap.add_argument("--routes", default="quad,one_thread,default,host")
    ap.add_argument("--label", default="")
    ap.add_argument("--no-rebuild", action="store_true")
    a = ap.parse_args()
    if not a.label:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        print("card:", q.stdout.strip().splitlines()[0] if q.stdout.strip() else "unknown", flush=True)
    routes = a.routes.split(",")
    dev = [r for r in routes if r != "host"]
    res = device_times(dev) if dev else {}
    if "host" in routes:
        res.update(host_times())
    for spec in a.compare:
        name, path = spec.split("=", 1)
        env = dict(os.environ, PORLA_TREE=os.path.abspath(path))
        print("--- %s (%s), default route" % (name, path), flush=True)
        subprocess.run([sys.executable, os.path.abspath(__file__), "--routes", "default", "--label", name, "--no-rebuild"],
                       env=env, check=True)
    if not a.no_rebuild:
        rebuild_side()


if __name__ == "__main__":
    main()
