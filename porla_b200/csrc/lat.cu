// Latency probe of the field / point operations for ONE block on ONE SM (development aid behind
// porla_debug_latency): how long a dependent chain of operations takes per operation when a warp has a
// scheduler to itself, and how much instruction-level parallelism between independent chains recovers.
// The small-MSM kernels (small_kernels.cuh), the bucket reduction below 2^18 points and the butterfly
// kernel all live in this regime.
//   mode 0  x = x * y                      one chain of Montgomery / special-form products
//   mode 1  two independent product chains in one thread
//   mode 2  four independent product chains in one thread
//   mode 3  x = x^2
//   mode 4  acc.add(q)    XYZZ + XYZZ, inlined field type
//   mode 5  acc.add(q)    XYZZ + XYZZ, outlined multiplier (FC)
//   mode 6  acc.madd(p)   XYZZ + affine, inlined
//   mode 7  acc = acc.dbl(), inlined
//   mode 8  x = 1/x + y    binary-GCD inversion (fp_inv.cuh);   mode 9: the same with the Fermat inversion
//   mode 10 / 11  quad_add / quad_dbl chains (quad.cuh: four lanes per point operation)
//   mode + 100: the same chain on the whole device (4 blocks per SM): ns_per_op is then the time per operation of a thread under load
// Measured (B200, BN254): 838 cycles per product with one warp per scheduler whether the thread runs one,
// two or four independent chains -- also with the two products interleaved round by round at source level
// (tried and removed) -- against ~600 cycles per product when two warps share a scheduler: the lone warp is
// bound by its own issue cadence on the multiplier pipe, not by the carry chains.
#include <cstdio>

#include "../../include/porla_multiexp.h"
#include "msm.h"
#include "msm_kernels.cuh"
#include "quad.cuh"

struct porla_table {   // as in staging.h
    porla::PointTable t;
};

namespace porla {

template <class C>
__global__ void k_latency(int mode, int iters, const Affine<typename C::F>* __restrict__ seed, unsigned long long* cycles,
                          XYZZ<typename C::F>* sink) {
    using F = typename C::F;
    using FC = typename C::FC;
    Affine<F> p = seed[threadIdx.x & 1];
    Affine<F> q = seed[2 + (threadIdx.x & 1)];
    XYZZ<F> acc = XYZZ<F>::from_affine(p);
    XYZZ<F> other = XYZZ<F>::from_affine(q);
    other = other.dbl();
    F x0 = p.x, x1 = p.y, x2 = q.x, x3 = q.y;
    const F y = q.y;
    __syncthreads();
    const long long t0 = clock64();
    if (mode == 0) {
#pragma unroll 1
        for (int i = 0; i < iters; i++) x0 = x0 * y;
    } else if (mode == 1) {
#pragma unroll 1
        for (int i = 0; i < iters; i++) {
            x0 = x0 * y;
            x1 = x1 * y;
        }
    } else if (mode == 2) {
#pragma unroll 1
        for (int i = 0; i < iters; i++) {
            x0 = x0 * y;
            x1 = x1 * y;
            x2 = x2 * y;
            x3 = x3 * y;
        }
    } else if (mode == 3) {
#pragma unroll 1
        for (int i = 0; i < iters; i++) x0 = x0.sqr();
    } else if (mode == 4) {
#pragma unroll 1
        for (int i = 0; i < iters; i++) acc.add(other);
    } else if (mode == 5) {
        XYZZ<FC> a2 = *reinterpret_cast<XYZZ<FC>*>(&acc), o2 = *reinterpret_cast<XYZZ<FC>*>(&other);
#pragma unroll 1
        for (int i = 0; i < iters; i++) a2.add(o2);
        acc = *reinterpret_cast<XYZZ<F>*>(&a2);
    } else if (mode == 6) {
#pragma unroll 1
        for (int i = 0; i < iters; i++) acc.madd_finite(q);
    } else if (mode == 7) {
#pragma unroll 1
        for (int i = 0; i < iters; i++) acc = acc.dbl();
    } else if (mode == 10 || mode == 11) {   // four lanes per point (quad.cuh): addition / doubling chains
        QuadPoint<F> qa = QuadPoint<F>::scatter(acc, 0), qo = QuadPoint<F>::scatter(other, 0);
        if (mode == 10) {
#pragma unroll 1
            for (int i = 0; i < iters; i++) qa = quad_add(qa, qo);
        } else {
#pragma unroll 1
            for (int i = 0; i < iters; i++) qa = quad_dbl(qa);
        }
        acc = qa.gather();
    } else if (mode == 8) {   // binary-GCD inversion (fp_inv.cuh), a dependent chain
#pragma unroll 1
        for (int i = 0; i < iters; i++) x0 = x0.inverse() + y;
    } else {                  // Fermat inversion, for comparison
#pragma unroll 1
        for (int i = 0; i < iters; i++) x0 = x0.inverse_fermat() + y;
    }
    const long long t1 = clock64();
    if (threadIdx.x % 32 == 0 && blockIdx.x == 0) cycles[threadIdx.x / 32] = (unsigned long long)(t1 - t0);
    acc.x = acc.x + x0 + x1 + x2 + x3;
    if (acc.x.v[0] == 0x12345678u && acc.y.v[1] == 0x9abcdef0u) *sink = acc;   // keep the work alive
}

// Parity harness of quad.cuh: out[i] = op(A_i, B_i), one quad per i (see porla_debug_quad_op).
template <class C>
__global__ void k_quad_op(int op, const Affine<typename C::F>* __restrict__ a, const Affine<typename C::F>* __restrict__ b, uint32_t n,
                          XYZZ<typename C::F>* __restrict__ out) {
    using F = typename C::F;
    const uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 2;
    const uint32_t j = i < n ? i : 0;
    QuadPoint<F> A = QuadPoint<F>::load_affine(a + j, false), B = QuadPoint<F>::load_affine(b + j, false);
    if (i >= n) A = B = QuadPoint<F>::inf();
    QuadPoint<F> r = QuadPoint<F>::inf();
    if (op == 0) r = quad_add(A, B);
    else if (op == 1) r = quad_dbl(A);
    else if (op == 2) r = quad_add(quad_dbl(A), quad_add(A, B));                  // 3A + B on general XYZZ operands
    else if (op == 3) {                                                            // 32 A through the P + P branch of quad_add
        r = A;
        for (int k = 0; k < 5; k++) r = quad_add(r, r);
    } else if (op == 4) r = quad_add(quad_add(A, B), QuadPoint<F>::load_affine(b + j, true));   // (A + B) - B = A, or inf cases
    else if (op == 5) {                                                            // scatter / gather round trip of the thread form
        XYZZ<F> t = XYZZ<F>::from_affine(ld16(a + j));
        t.madd(ld16(b + j));
        r = QuadPoint<F>::scatter(t, (int)(i & 3));
        XYZZ<F> g = r.gather();
        g = g.dbl();
        r = QuadPoint<F>::scatter(g, (int)((i + 1) & 3));                          // 2 (A + B)
    }
    if (i < n) r.store(out + i);
}

}  // namespace porla

// out64[i] (affine, external bytes) = op(A_i, B_i) computed with the four-lane point operations of quad.cuh:
// op 0: A + B, 1: 2A, 2: 3A + B, 3: 32A, 4: (A + B) - B, 5: 2 (A + B) through scatter / gather.
extern "C" void porla_debug_quad_op(int curve, int op, const porla_table* a, const porla_table* b, int64_t n, int point_fmt, void* out64) {
    using namespace porla;
    device_init();
    void* d_x = nullptr;
    uint8_t* d_out = nullptr;
    PORLA_CUDA(cudaMalloc(&d_x, (size_t)n * 128 + 128));
    PORLA_CUDA(cudaMalloc(&d_out, (size_t)n * 64 + 64));
    const uint32_t threads = (uint32_t)n * 4, blocks = (threads + 127) / 128;
    if (curve == kCurveBn254) {
        k_quad_op<Bn254><<<blocks, 128>>>(op, reinterpret_cast<const Affine<Bn254::F>*>(a->t.d_points),
                                          reinterpret_cast<const Affine<Bn254::F>*>(b->t.d_points), (uint32_t)n, reinterpret_cast<XYZZ<Bn254::F>*>(d_x));
        k_finalize<Bn254><<<((uint32_t)n + 31) / 32, 32>>>(reinterpret_cast<const XYZZ<Bn254::FC>*>(d_x), (uint32_t)n, 1, 1, point_fmt, d_out, nullptr);
    } else {
        k_quad_op<Secp256k1><<<blocks, 128>>>(op, reinterpret_cast<const Affine<Secp256k1::F>*>(a->t.d_points),
                                              reinterpret_cast<const Affine<Secp256k1::F>*>(b->t.d_points), (uint32_t)n,
                                              reinterpret_cast<XYZZ<Secp256k1::F>*>(d_x));
        k_finalize<Secp256k1><<<((uint32_t)n + 31) / 32, 32>>>(reinterpret_cast<const XYZZ<Secp256k1::FC>*>(d_x), (uint32_t)n, 1, 1, point_fmt, d_out,
                                                               nullptr);
    }
    PORLA_CUDA(cudaGetLastError());
    PORLA_CUDA(cudaMemcpy(out64, d_out, (size_t)n * 64, cudaMemcpyDeviceToHost));
    PORLA_CUDA(cudaFree(d_x));
    PORLA_CUDA(cudaFree(d_out));
}

extern "C" int porla_debug_latency(int curve, int mode, int warps, int iters, double* cycles_per_op, double* ns_per_op) {
    using namespace porla;
    device_init();
    // mode + 100: the same chain in `warps` warps per block on 4 blocks per SM of the whole device (throughput under load)
    int blocks = 1;
    if (mode >= 100) {
        mode -= 100;
        cudaDeviceProp prop;
        int dev = 0;
        PORLA_CUDA(cudaGetDevice(&dev));
        PORLA_CUDA(cudaGetDeviceProperties(&prop, dev));
        blocks = prop.multiProcessorCount * 4;
    }
    if (warps < 1) warps = 1;
    if (warps > 32) warps = 32;
    // four affine points: small multiples of the generator, built on the host side of the library
    porla_table* t = nullptr;
    uint32_t ks[4][8] = {{3}, {5}, {7}, {11}};
    t = porla_table_create_multiples(curve, ks, 4, PORLA_SCALAR_LE32, 0, nullptr);
    unsigned long long* d_cycles = nullptr;
    void* d_sink = nullptr;
    PORLA_CUDA(cudaMalloc(&d_cycles, 32 * 8));
    PORLA_CUDA(cudaMalloc(&d_sink, 256));
    cudaEvent_t e0, e1;
    PORLA_CUDA(cudaEventCreate(&e0));
    PORLA_CUDA(cudaEventCreate(&e1));
    const void* pts = t->t.d_points;
    float ms = 0;
    for (int rep = 0; rep < 3; rep++) {
        PORLA_CUDA(cudaEventRecord(e0));
        if (curve == kCurveBn254)
            k_latency<Bn254><<<blocks, warps * 32>>>(mode, iters, reinterpret_cast<const Affine<Bn254::F>*>(pts), d_cycles,
                                               reinterpret_cast<XYZZ<Bn254::F>*>(d_sink));
        else
            k_latency<Secp256k1><<<blocks, warps * 32>>>(mode, iters, reinterpret_cast<const Affine<Secp256k1::F>*>(pts), d_cycles,
                                                   reinterpret_cast<XYZZ<Secp256k1::F>*>(d_sink));
        PORLA_CUDA(cudaEventRecord(e1));
        PORLA_CUDA(cudaEventSynchronize(e1));
        PORLA_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    }
    unsigned long long h[32] = {};
    PORLA_CUDA(cudaMemcpy(h, d_cycles, (size_t)warps * 8, cudaMemcpyDeviceToHost));
    unsigned long long mx = 0;
    for (int w = 0; w < warps; w++) mx = h[w] > mx ? h[w] : mx;
    const double ops = (double)iters * (mode == 1 ? 2.0 : mode == 2 ? 4.0 : 1.0);
    *cycles_per_op = (double)mx / ops;
    *ns_per_op = (double)ms * 1e6 / ops;
    PORLA_CUDA(cudaEventDestroy(e0));
    PORLA_CUDA(cudaEventDestroy(e1));
    PORLA_CUDA(cudaFree(d_cycles));
    PORLA_CUDA(cudaFree(d_sink));
    porla_table_destroy(t);
    return 0;
}
