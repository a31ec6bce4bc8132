"""Workload for compute-sanitizer (memcheck / racecheck): touches every kernel of the pipeline once,
including the shared-memory radix partition (n >= 2^19) and the batched / fixed-base / butterfly paths."""
import os, sys, random
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import porla_b200 as pb
from oracle import curves_py as O
be = lambda v: v.to_bytes(32, "big")
lib = pb.load(); lib.porla_device_init()
g = torch.Generator(device="cuda"); g.manual_seed(3)
big = os.environ.get("SAN_BIG", "1") == "1"
for curve in (pb.CURVE_BN254, pb.CURVE_SECP256K1):
    n = (1 << 19) + 37 if big else 5000
    ks = torch.randint(0, 2**15, (n, 8), dtype=torch.int32, device="cuda", generator=g)
    ks[:, 1:] = 0
    ks[5::7] = 0
    tab = pb.Table.multiples_of_generator(curve, ks.data_ptr(), n, pb.SCALAR_LE32, on_device=True)
    ss = torch.randint(-2**31, 2**31 - 1, (n, 8), dtype=torch.int32, device="cuda", generator=g)
    a = tab.msm_resident(ss.data_ptr(), n, scalar_fmt=pb.SCALAR_LE32)
    ss[:] = ss[0]
    b = tab.msm_resident(ss.data_ptr(), n, scalar_fmt=pb.SCALAR_LE32)      # constant scalar: long stitch
    out = torch.zeros(64 * 8, dtype=torch.uint8, device="cuda")
    tab.msm_device(ss.data_ptr(), 600, out.data_ptr(), nbatch=8, scalar_fmt=pb.SCALAR_LE32, shared_points=True)
    tab2 = pb.Table.multiples_of_generator(curve, ks.data_ptr(), 256, pb.SCALAR_LE32, on_device=True)
    tab2.precompute(0, 256, 8)
    tab2.msm_device(ss.data_ptr(), 256, out.data_ptr(), nbatch=8, scalar_fmt=pb.SCALAR_LE32, shared_points=True)
    tab2.butterfly_stage(4, be(3) + be(5))
    torch.cuda.synchronize()
    print("curve", curve, a.hex()[:16], b.hex()[:16], flush=True)
    tab.destroy(); tab2.destroy()
k = pb.Kzg(bytes.fromhex("ffeeddccbbaa99887766554433221100"), bytes.fromhex("00112233445566778899aabbccddeeff"))
k.init_srs(32)
rnd = random.Random(1)
data = bytearray(b"".join(rnd.randrange(1 << 500).to_bytes(64, "little") for _ in range(32 * 3)))
print("align", k.align_mac_batch(data, 3).hex()[:16])
print("proof", k.create_proof(77, b"".join(be(rnd.randrange(1 << 256)) for _ in range(32)))[0].hex()[:16])
# one-launch small paths: bitwise tree sum (1 and several blocks per window, batched), look-up-table sums (single,
# batch with one scalar per thread), sub-range view of the table, block aggregation of an audit
coeff = b"".join(pb.bn254_scalar_set_int(rnd.randrange(1 << 31)) for _ in range(700))
G = O.bn254_marshal((1, 2))
pts = G * 700
print("bits", pb.bn254_multi_exp(pts, coeff, 700).hex()[:16], pb.bn254_multi_exp(pts[:64 * 100], coeff[:32 * 100], 100).hex()[:16])
print("bits batch", pb.bn254_multi_exp_batch(pts[:64 * 120], coeff[:32 * 120], 40, 3).hex()[:16])
blocks = b"".join(be(rnd.randrange(1 << 256)) for _ in range(32 * 20))
print("lut", k.compute_digest_from_srs(blocks[:32 * 32]).hex()[:16], k.compute_digest_from_srs_batch(blocks, 20).hex()[:16])
cf = b"".join(rnd.randrange(1 << 31).to_bytes(4, "little") for _ in range(50))
bl = b"".join(rnd.randrange(1 << 500).to_bytes(64, "little") for _ in range(50 * 32))
print("aggregate", k.audit_aggregate(cf, bl, 50)[1].hex()[:16])
c = O.SECP256K1
gens = pb.SecpGenerators([(c.gx, c.gy)] * 64)
print("secp lut", gens.multi(0, [rnd.randrange(c.n) for _ in range(64)])[0], gens.multi(16, [rnd.randrange(c.n) for _ in range(16)])[0])
gens.destroy()
# IPA prover and verifier over generators + u (batch of two look-up sums per round, 12-point variable-base MSM)
pts = [O.mul(c, k_, (c.gx, c.gy)) for k_ in range(2, 19)]
gu = pb.SecpGenerators(pts)
a_, b_ = [rnd.randrange(c.n) for _ in range(16)], [rnd.randrange(c.n) for _ in range(16)]
pr = gu.inner_product_prove(a_, b_)
print("ipa", len(pr), gu.inner_product_verify(O.msm(c, a_, pts[:16]), pr))
gu.destroy()
# data-side FFT stage
import ctypes as C
LCM = (207 * 2**248 + 1) * O.BN254.n
blk = bytearray(b"".join(rnd.randrange(LCM).to_bytes(64, "little") for _ in range(8 * 5)))
lib.porla_data_butterfly_stage(C.cast((C.c_ubyte * len(blk)).from_buffer(blk), C.c_void_p), 8, 5, 4,
                               b"".join(rnd.randrange(1 << 256).to_bytes(32, "little") for _ in range(2)), LCM.to_bytes(64, "little"))
print("data fft", bytes(blk[:8]).hex())
# round 2: streamed host-buffer MSM (parts accumulated into one bucket set), in-call partition over several workers, sharded
# resident table, affine accumulation kernel, batched scalar multiplication, device butterfly stage forced
from oracle import loader
os.environ["PORLA_OVERSUBSCRIBE_DEVICES"] = "1"
n = 6000
G = O.bn254_marshal((1, 2)); step = O.bn254_marshal(O.mul(O.BN254, 0xC0FFEE, (1, 2)))
hp = bytearray(loader.bn254_point_chain(G, step, n)); hp[64 * 9:64 * 10] = bytes(64)
hs = b"".join(be(rnd.randrange(1 << 256)) for _ in range(n))
os.environ["PORLA_STREAM_PARTS"] = "3"
r1 = pb.msm_host_devices(pb.CURVE_BN254, hs, bytes(hp), n, 1)
r2 = pb.msm_host_devices(pb.CURVE_BN254, hs, bytes(hp), n, 3)
del os.environ["PORLA_STREAM_PARTS"]
mt = pb.MultiTable(pb.CURVE_BN254, bytes(hp), n, ndev=3)
r3 = mt.msm_host_scalars(hs)
ptrs = mt.upload_scalars(hs); r4 = mt.msm_resident(ptrs); mt.free_scalars(ptrs); mt.destroy()
print("streamed / fan-out / sharded table:", r1 == r2 == r3 == r4, r1.hex()[:16])
# round 2c: the old bucket reduction, the fixed-base sharded form, the four-lane point operations' parity harness
os.environ["PORLA_REDUCE_V1"] = "1"; os.environ["PORLA_NO_SMALL"] = "1"
r7 = pb.bn254_multi_exp(bytes(hp), hs, n)
del os.environ["PORLA_REDUCE_V1"]; del os.environ["PORLA_NO_SMALL"]
tfb = pb.Table.from_host(pb.CURVE_BN254, bytes(hp)); cfb = tfb.precompute(12, n, 1)
d_hs = torch.frombuffer(bytearray(hs), dtype=torch.uint8).cuda(); d_ws = torch.zeros(128, dtype=torch.uint8, device="cuda")
code = cfb | pb.lib.PLAN_FIXED | pb.lib.PLAN_GLV_OFF
lib.porla_msm_window_sums_device(C.c_void_p(tfb.handle), C.c_void_p(d_hs.data_ptr()), n, pb.SCALAR_BE32, code, C.c_void_p(d_ws.data_ptr()), None)
torch.cuda.synchronize()
o64 = (C.c_ubyte * 64)()
lib.porla_msm_finalize_host(pb.CURVE_BN254, d_ws.cpu().numpy().tobytes(), 1, 1, code, pb.POINT_BE64, C.cast(o64, C.c_void_p))
r8 = bytes(o64)
oq = (C.c_ubyte * (64 * 40))()
for op in range(6):
    lib.porla_debug_quad_op(pb.CURVE_BN254, op, C.c_void_p(tfb.handle), C.c_void_p(tfb.handle), 40, pb.POINT_BE64, oq)
tfb.destroy()
print("old reduce / fixed-base sharded form:", r1 == r7 == r8)
tabs = pb.Table.from_host(pb.CURVE_BN254, bytes(hp[:64 * 40]))
d_sc = torch.frombuffer(bytearray(hs[:32 * 40]), dtype=torch.uint8).cuda()
d_out = torch.zeros(64 * 40, dtype=torch.uint8, device="cuda")
lib.porla_scalar_mul_batch_device(C.c_void_p(tabs.handle), C.c_void_p(d_sc.data_ptr()), 40, pb.SCALAR_BE32, pb.POINT_BE64,
                                  C.c_void_p(d_out.data_ptr()), None)
torch.cuda.synchronize(); tabs.destroy()
os.environ["PORLA_HOST_BUTTERFLIES"] = "0"
buf = bytearray(hp[:64 * 16]); pb.bn254_butterfly_stage(buf, 16, 4, be(7) + be(9))
del os.environ["PORLA_HOST_BUTTERFLIES"]
print("scalar mul batch / device butterfly", bytes(buf[:8]).hex())
print("done")
