// 256-bit prime-field arithmetic on 8 x 32-bit limbs for sm_100a (and a portable host path).
//
// Two reduction families, selected by the parameter struct:
//   * Montgomery CIOS for BN254 Fp (p < 2^254, two spare bits => no extra carry limb), replacing
//     gnark-crypto's 4x64 Montgomery `fp.Element` that /root/reference/porla/main.go reaches
//     through bn254.G1Affine (main.go:130,136).
//   * Special-form fold for secp256k1 Fp (p = 2^256 - 2^32 - 977), replacing the 5x52 + __int128
//     code of /root/reference/porla/Utils/secp256k1_lib/field_5x52_int128_impl.h:18.
//
// Device path: inline-PTX carry chains.  Products are accumulated in two interleaved
// "even"/"odd" rows so that every 32x32->64 product lands on a 64-bit aligned slot; ptxas
// turns each mad.lo.cc/madc.hi.cc pair into one IMAD.WIDE.U32(.X) (checked with cuobjdump).
// Host path (no __CUDA_ARCH__): plain uint64_t arithmetic, used by the C-ABI's single-point
// operations and by the CPU-side unit tests of the formulas.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define PORLA_HD __host__ __device__ __forceinline__
#define PORLA_D __device__ __forceinline__
#else
#define PORLA_HD inline
#define PORLA_D inline
#endif

namespace porla {

// ------------------------------------------------------------------------------------------
// Parameter packs.  Constants are returned through switch-free constexpr lookups so that fully
// unrolled code sees immediates.
// ------------------------------------------------------------------------------------------
struct Bn254FpParams {
    static constexpr bool kMontgomery = true;
    // p = 21888242871839275222246405745257275088696311157297823662689037894645226208583
    PORLA_HD static constexpr uint32_t mod(int i) {
        constexpr uint32_t m[8] = {0xd87cfd47u, 0x3c208c16u, 0x6871ca8du, 0x97816a91u,
                                   0x8181585du, 0xb85045b6u, 0xe131a029u, 0x30644e72u};
        return m[i];
    }
    // R^2 mod p, R = 2^256
    PORLA_HD static constexpr uint32_t r2(int i) {
        constexpr uint32_t m[8] = {0x538afa89u, 0xf32cfc5bu, 0xd44501fbu, 0xb5e71911u,
                                   0x0a417ff6u, 0x47ab1effu, 0xcab8351fu, 0x06d89f71u};
        return m[i];
    }
    // R mod p (Montgomery one)
    PORLA_HD static constexpr uint32_t one(int i) {
        constexpr uint32_t m[8] = {0xc58f0d9du, 0xd35d438du, 0xf5c70b3du, 0x0a78eb28u,
                                   0x7879462cu, 0x666ea36fu, 0x9a07df2fu, 0x0e0a77c1u};
        return m[i];
    }
    static constexpr uint32_t kInv = 0xe4866389u;  // -p^{-1} mod 2^32
    static constexpr int kBits = 254;
};

// BN254 scalar field Fr (order of G1); used on the host for KZG polynomial arithmetic
// (polynomial.Eval, kzg.Open in /root/reference/porla/main.go:81,170).
struct Bn254FrParams {
    static constexpr bool kMontgomery = true;
    PORLA_HD static constexpr uint32_t mod(int i) {
        constexpr uint32_t m[8] = {0xf0000001u, 0x43e1f593u, 0x79b97091u, 0x2833e848u,
                                   0x8181585du, 0xb85045b6u, 0xe131a029u, 0x30644e72u};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t r2(int i) {
        constexpr uint32_t m[8] = {0xae216da7u, 0x1bb8e645u, 0xe35c59e3u, 0x53fe3ab1u,
                                   0x53bb8085u, 0x8c49833du, 0x7f4e44a5u, 0x0216d0b1u};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t one(int i) {
        constexpr uint32_t m[8] = {0x4ffffffbu, 0xac96341cu, 0x9f60cd29u, 0x36fc7695u,
                                   0x7879462eu, 0x666ea36fu, 0x9a07df2fu, 0x0e0a77c1u};
        return m[i];
    }
    static constexpr uint32_t kInv = 0xefffffffu;
    static constexpr int kBits = 254;
};

struct Secp256k1FpParams {
    static constexpr bool kMontgomery = false;
    // p = 2^256 - 2^32 - 977
    PORLA_HD static constexpr uint32_t mod(int i) {
        constexpr uint32_t m[8] = {0xfffffc2fu, 0xfffffffeu, 0xffffffffu, 0xffffffffu,
                                   0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t one(int i) { return i == 0 ? 1u : 0u; }
    PORLA_HD static constexpr uint32_t r2(int i) { return i == 0 ? 1u : 0u; }
    static constexpr uint32_t kInv = 0;
    static constexpr int kBits = 256;
};

// ------------------------------------------------------------------------------------------
// Raw 256-bit helpers (shared by base fields and by scalar recoding).
// ------------------------------------------------------------------------------------------
// r = a + b, returns carry
PORLA_HD uint32_t add256(uint32_t* r, const uint32_t* a, const uint32_t* b) {
#ifdef __CUDA_ARCH__
    uint32_t c;
    asm("add.cc.u32 %0, %9, %17;\n\t"
        "addc.cc.u32 %1, %10, %18;\n\t"
        "addc.cc.u32 %2, %11, %19;\n\t"
        "addc.cc.u32 %3, %12, %20;\n\t"
        "addc.cc.u32 %4, %13, %21;\n\t"
        "addc.cc.u32 %5, %14, %22;\n\t"
        "addc.cc.u32 %6, %15, %23;\n\t"
        "addc.cc.u32 %7, %16, %24;\n\t"
        "addc.u32 %8, 0, 0;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
          "=r"(r[7]), "=r"(c)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
    return c;
#else
    uint64_t c = 0;
    for (int i = 0; i < 8; i++) {
        c += (uint64_t)a[i] + b[i];
        r[i] = (uint32_t)c;
        c >>= 32;
    }
    return (uint32_t)c;
#endif
}

// r = a - b, returns borrow (1 if a < b)
PORLA_HD uint32_t sub256(uint32_t* r, const uint32_t* a, const uint32_t* b) {
#ifdef __CUDA_ARCH__
    uint32_t c;
    asm("sub.cc.u32 %0, %9, %17;\n\t"
        "subc.cc.u32 %1, %10, %18;\n\t"
        "subc.cc.u32 %2, %11, %19;\n\t"
        "subc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\t"
        "subc.cc.u32 %5, %14, %22;\n\t"
        "subc.cc.u32 %6, %15, %23;\n\t"
        "subc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
          "=r"(r[7]), "=r"(c)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
    return c & 1u;
#else
    int64_t c = 0;
    for (int i = 0; i < 8; i++) {
        c += (int64_t)a[i] - (int64_t)b[i];
        r[i] = (uint32_t)c;
        c >>= 32;
    }
    return (uint32_t)(c & 1);
#endif
}


}  // namespace porla
#include "fp_inv.cuh"
namespace porla {

#ifdef __CUDA_ARCH__
// ------------------------------------------------------------------------------------------
// Carry-chain building blocks (device).  r points at 2k consecutive 32-bit accumulator limbs that
// start on a 64-bit aligned slot of their row; every mad.lo.cc/madc.hi.cc pair becomes one
// IMAD.WIDE.U32(.X).  `top` is the limb right above the chain and receives the carry-out.
// ------------------------------------------------------------------------------------------
PORLA_D void mac4(uint32_t* r, uint32_t& top, uint32_t x0, uint32_t x1, uint32_t x2, uint32_t x3, uint32_t s) {
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t"
        "madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
        "madc.lo.cc.u32 %2, %10, %13, %2;\n\t"
        "madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\t"
        "madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
        "madc.lo.cc.u32 %6, %12, %13, %6;\n\t"
        "madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
        "addc.u32 %8, %8, 0;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(top)
        : "r"(x0), "r"(x1), "r"(x2), "r"(x3), "r"(s));
}
PORLA_D void mac3(uint32_t* r, uint32_t& top, uint32_t x0, uint32_t x1, uint32_t x2, uint32_t s) {
    asm("mad.lo.cc.u32 %0, %7, %10, %0;\n\t"
        "madc.hi.cc.u32 %1, %7, %10, %1;\n\t"
        "madc.lo.cc.u32 %2, %8, %10, %2;\n\t"
        "madc.hi.cc.u32 %3, %8, %10, %3;\n\t"
        "madc.lo.cc.u32 %4, %9, %10, %4;\n\t"
        "madc.hi.cc.u32 %5, %9, %10, %5;\n\t"
        "addc.u32 %6, %6, 0;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(top)
        : "r"(x0), "r"(x1), "r"(x2), "r"(s));
}
PORLA_D void mac2(uint32_t* r, uint32_t& top, uint32_t x0, uint32_t x1, uint32_t s) {
    asm("mad.lo.cc.u32 %0, %5, %7, %0;\n\t"
        "madc.hi.cc.u32 %1, %5, %7, %1;\n\t"
        "madc.lo.cc.u32 %2, %6, %7, %2;\n\t"
        "madc.hi.cc.u32 %3, %6, %7, %3;\n\t"
        "addc.u32 %4, %4, 0;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(top)
        : "r"(x0), "r"(x1), "r"(s));
}
PORLA_D void mac1(uint32_t* r, uint32_t& top, uint32_t x0, uint32_t s) {
    asm("mad.lo.cc.u32 %0, %3, %4, %0;\n\t"
        "madc.hi.cc.u32 %1, %3, %4, %1;\n\t"
        "addc.u32 %2, %2, 0;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(top)
        : "r"(x0), "r"(s));
}

// T[0..15] = a * b, schoolbook on two rows: E holds the products that land on even limbs
// (E[k] = limb k), O those on odd limbs (O[k] = limb k + 1).  Row i's carry-out goes to a limb that
// so far holds nothing but earlier carry-outs, so no carry ever ripples further.
PORLA_D void mul_wide_device(const uint32_t* a, const uint32_t* b, uint32_t* T) {
    uint32_t E[16], O[16];
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
        uint64_t pe = (uint64_t)a[j] * b[0], po = (uint64_t)a[j + 1] * b[0];
        E[j] = (uint32_t)pe;
        E[j + 1] = (uint32_t)(pe >> 32);
        O[j] = (uint32_t)po;
        O[j + 1] = (uint32_t)(po >> 32);
    }
#pragma unroll
    for (int j = 8; j < 16; j++) E[j] = O[j] = 0;
#pragma unroll
    for (int i = 1; i < 8; i++) {
        if (i & 1) {
            if (i + 9 < 16) mac4(E + i + 1, E[i + 9], a[1], a[3], a[5], a[7], b[i]);
            else { uint32_t drop = 0; mac4(E + i + 1, drop, a[1], a[3], a[5], a[7], b[i]); }
            mac4(O + i - 1, O[i + 7], a[0], a[2], a[4], a[6], b[i]);
        } else {
            mac4(E + i, E[i + 8], a[0], a[2], a[4], a[6], b[i]);
            mac4(O + i, O[i + 8], a[1], a[3], a[5], a[7], b[i]);
        }
    }
    T[0] = E[0];
    asm("add.cc.u32 %0, %15, %30;\n\t"
        "addc.cc.u32 %1, %16, %31;\n\t"
        "addc.cc.u32 %2, %17, %32;\n\t"
        "addc.cc.u32 %3, %18, %33;\n\t"
        "addc.cc.u32 %4, %19, %34;\n\t"
        "addc.cc.u32 %5, %20, %35;\n\t"
        "addc.cc.u32 %6, %21, %36;\n\t"
        "addc.cc.u32 %7, %22, %37;\n\t"
        "addc.cc.u32 %8, %23, %38;\n\t"
        "addc.cc.u32 %9, %24, %39;\n\t"
        "addc.cc.u32 %10, %25, %40;\n\t"
        "addc.cc.u32 %11, %26, %41;\n\t"
        "addc.cc.u32 %12, %27, %42;\n\t"
        "addc.cc.u32 %13, %28, %43;\n\t"
        "addc.u32 %14, %29, %44;"
        : "=r"(T[1]), "=r"(T[2]), "=r"(T[3]), "=r"(T[4]), "=r"(T[5]), "=r"(T[6]), "=r"(T[7]), "=r"(T[8]),
          "=r"(T[9]), "=r"(T[10]), "=r"(T[11]), "=r"(T[12]), "=r"(T[13]), "=r"(T[14]), "=r"(T[15])
        : "r"(E[1]), "r"(E[2]), "r"(E[3]), "r"(E[4]), "r"(E[5]), "r"(E[6]), "r"(E[7]), "r"(E[8]), "r"(E[9]),
          "r"(E[10]), "r"(E[11]), "r"(E[12]), "r"(E[13]), "r"(E[14]), "r"(E[15]),
          "r"(O[0]), "r"(O[1]), "r"(O[2]), "r"(O[3]), "r"(O[4]), "r"(O[5]), "r"(O[6]), "r"(O[7]), "r"(O[8]),
          "r"(O[9]), "r"(O[10]), "r"(O[11]), "r"(O[12]), "r"(O[13]), "r"(O[14]));
}

// T[0..15] = a^2: the 28 off-diagonal products once (same two-row scheme), doubled, plus the 8
// squares a_i^2 in one chain: 36 multiplies instead of 64.
PORLA_D void sqr_wide_device(const uint32_t* a, uint32_t* T) {
    uint32_t E[16], O[16];  // E[k] = limb k (even-sum products), O[k] = limb k + 1 (odd-sum products)
#pragma unroll
    for (int j = 0; j < 16; j++) E[j] = O[j] = 0;
    // odd sums i + j: chains start at limb 2i + 1 = O[2i]
    mac4(O + 0, O[8], a[1], a[3], a[5], a[7], a[0]);    // (0,1) (0,3) (0,5) (0,7)
    mac3(O + 2, O[8], a[2], a[4], a[6], a[1]);          // (1,2) (1,4) (1,6)
    mac3(O + 4, O[10], a[3], a[5], a[7], a[2]);         // (2,3) (2,5) (2,7)
    mac2(O + 6, O[10], a[4], a[6], a[3]);               // (3,4) (3,6)
    mac2(O + 8, O[12], a[5], a[7], a[4]);               // (4,5) (4,7)
    mac1(O + 10, O[12], a[6], a[5]);                    // (5,6)
    mac1(O + 12, O[14], a[7], a[6]);                    // (6,7)
    // even sums: chains start at limb 2i + 2 = E[2i + 2]
    mac3(E + 2, E[8], a[2], a[4], a[6], a[0]);          // (0,2) (0,4) (0,6)
    mac3(E + 4, E[10], a[3], a[5], a[7], a[1]);         // (1,3) (1,5) (1,7)
    mac2(E + 6, E[10], a[4], a[6], a[2]);               // (2,4) (2,6)
    mac2(E + 8, E[12], a[5], a[7], a[3]);               // (3,5) (3,7)
    mac1(E + 10, E[12], a[6], a[4]);                    // (4,6)
    mac1(E + 12, E[14], a[7], a[5]);                    // (5,7)
    // S = E + (O << 32)   (limbs 1..15; limb 0 of the off-diagonal sum is zero)
    uint32_t S[16];
    S[0] = 0;
    asm("add.cc.u32 %0, %15, %30;\n\t"
        "addc.cc.u32 %1, %16, %31;\n\t"
        "addc.cc.u32 %2, %17, %32;\n\t"
        "addc.cc.u32 %3, %18, %33;\n\t"
        "addc.cc.u32 %4, %19, %34;\n\t"
        "addc.cc.u32 %5, %20, %35;\n\t"
        "addc.cc.u32 %6, %21, %36;\n\t"
        "addc.cc.u32 %7, %22, %37;\n\t"
        "addc.cc.u32 %8, %23, %38;\n\t"
        "addc.cc.u32 %9, %24, %39;\n\t"
        "addc.cc.u32 %10, %25, %40;\n\t"
        "addc.cc.u32 %11, %26, %41;\n\t"
        "addc.cc.u32 %12, %27, %42;\n\t"
        "addc.cc.u32 %13, %28, %43;\n\t"
        "addc.u32 %14, %29, %44;"
        : "=r"(S[1]), "=r"(S[2]), "=r"(S[3]), "=r"(S[4]), "=r"(S[5]), "=r"(S[6]), "=r"(S[7]), "=r"(S[8]),
          "=r"(S[9]), "=r"(S[10]), "=r"(S[11]), "=r"(S[12]), "=r"(S[13]), "=r"(S[14]), "=r"(S[15])
        : "r"(E[1]), "r"(E[2]), "r"(E[3]), "r"(E[4]), "r"(E[5]), "r"(E[6]), "r"(E[7]), "r"(E[8]), "r"(E[9]),
          "r"(E[10]), "r"(E[11]), "r"(E[12]), "r"(E[13]), "r"(E[14]), "r"(E[15]),
          "r"(O[0]), "r"(O[1]), "r"(O[2]), "r"(O[3]), "r"(O[4]), "r"(O[5]), "r"(O[6]), "r"(O[7]), "r"(O[8]),
          "r"(O[9]), "r"(O[10]), "r"(O[11]), "r"(O[12]), "r"(O[13]), "r"(O[14]));
    // T = 2 S  (funnel shifts; S < 2^511)
#pragma unroll
    for (int k = 15; k > 0; k--) T[k] = __funnelshift_l(S[k - 1], S[k], 1);
    T[0] = 0;
    // T += sum a_i^2 * 2^(64 i): one 16-limb chain
    asm("mad.lo.cc.u32 %0, %16, %16, %0;\n\t"
        "madc.hi.cc.u32 %1, %16, %16, %1;\n\t"
        "madc.lo.cc.u32 %2, %17, %17, %2;\n\t"
        "madc.hi.cc.u32 %3, %17, %17, %3;\n\t"
        "madc.lo.cc.u32 %4, %18, %18, %4;\n\t"
        "madc.hi.cc.u32 %5, %18, %18, %5;\n\t"
        "madc.lo.cc.u32 %6, %19, %19, %6;\n\t"
        "madc.hi.cc.u32 %7, %19, %19, %7;\n\t"
        "madc.lo.cc.u32 %8, %20, %20, %8;\n\t"
        "madc.hi.cc.u32 %9, %20, %20, %9;\n\t"
        "madc.lo.cc.u32 %10, %21, %21, %10;\n\t"
        "madc.hi.cc.u32 %11, %21, %21, %11;\n\t"
        "madc.lo.cc.u32 %12, %22, %22, %12;\n\t"
        "madc.hi.cc.u32 %13, %22, %22, %13;\n\t"
        "madc.lo.cc.u32 %14, %23, %23, %14;\n\t"
        "madc.hi.u32 %15, %23, %23, %15;"
        : "+r"(T[0]), "+r"(T[1]), "+r"(T[2]), "+r"(T[3]), "+r"(T[4]), "+r"(T[5]), "+r"(T[6]), "+r"(T[7]),
          "+r"(T[8]), "+r"(T[9]), "+r"(T[10]), "+r"(T[11]), "+r"(T[12]), "+r"(T[13]), "+r"(T[14]), "+r"(T[15])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]));
}
#endif  // __CUDA_ARCH__

// ------------------------------------------------------------------------------------------
// Field element
// ------------------------------------------------------------------------------------------
// kCompact = true routes every device-side product through ONE non-inlined copy of the multiplier
// (8 + 8 registers in, 8 out).  The bucket-accumulation kernel wants everything inlined; the cold
// kernels (bucket reduction, stitching, window combine) inline a dozen XYZZ additions and become
// instruction-fetch bound (ncu: stall_no_instruction dominates) unless the code is kept small.
template <class P, bool kCompact>
struct Fp;
#ifdef __CUDACC__
template <class P>
__device__ __noinline__ Fp<P, true> fp_mul_outlined(Fp<P, true> a, Fp<P, true> b);
#endif

template <class P, bool kCompact = false>
struct alignas(16) Fp {
    uint32_t v[8];
    using Params = P;

    PORLA_HD static Fp zero() {
        Fp r;
#pragma unroll
        for (int i = 0; i < 8; i++) r.v[i] = 0;
        return r;
    }
    PORLA_HD static Fp one() {
        Fp r;
#pragma unroll
        for (int i = 0; i < 8; i++) r.v[i] = P::one(i);
        return r;
    }
    PORLA_HD static Fp modulus() {
        Fp r;
#pragma unroll
        for (int i = 0; i < 8; i++) r.v[i] = P::mod(i);
        return r;
    }
    PORLA_HD bool is_zero() const {
        uint32_t o = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) o |= v[i];
        return o == 0;
    }
    PORLA_HD bool operator==(const Fp& b) const {
        uint32_t o = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) o |= v[i] ^ b.v[i];
        return o == 0;
    }
    PORLA_HD bool operator!=(const Fp& b) const { return !(*this == b); }

    // canonical reduce of a value known to be < 2p (carry = bit 256 of the value)
    PORLA_HD void final_sub(uint32_t carry) {
        uint32_t t[8], m[8];
#pragma unroll
        for (int i = 0; i < 8; i++) m[i] = P::mod(i);
        uint32_t borrow = sub256(t, v, m);
        // value >= p  <=>  carry || !borrow
        bool take = carry | (borrow ^ 1u);
#pragma unroll
        for (int i = 0; i < 8; i++) v[i] = take ? t[i] : v[i];
    }

    PORLA_HD friend Fp operator+(const Fp& a, const Fp& b) {
        Fp r;
        uint32_t c = add256(r.v, a.v, b.v);
        r.final_sub(c);
        return r;
    }
    PORLA_HD friend Fp operator-(const Fp& a, const Fp& b) {
        Fp r;
        uint32_t borrow = sub256(r.v, a.v, b.v);
        uint32_t t[8], m[8];
#pragma unroll
        for (int i = 0; i < 8; i++) m[i] = P::mod(i);
        add256(t, r.v, m);
#pragma unroll
        for (int i = 0; i < 8; i++) r.v[i] = borrow ? t[i] : r.v[i];
        return r;
    }
    PORLA_HD Fp neg() const {
        Fp r;
        uint32_t m[8];
#pragma unroll
        for (int i = 0; i < 8; i++) m[i] = P::mod(i);
        sub256(r.v, m, v);
        bool z = is_zero();
#pragma unroll
        for (int i = 0; i < 8; i++) r.v[i] = z ? 0u : r.v[i];
        return r;
    }
    PORLA_HD Fp dbl() const { return *this + *this; }

    // -------------------------------------------------------------------------- multiplication
#ifdef __CUDA_ARCH__
    // One CIOS round of the even/odd-row Montgomery product (see mul_mont_device below).
    // Invariant on entry (round >= 1):  T = E + O[1]*2^0 + sum_{k<6} O[k+2]*2^(32(k+1)),
    // i.e. O is the row that was reduced in the previous round (O[0] == 0) viewed one limb lower.
    // Each carry chain lives inside ONE asm statement so the compiler cannot split it.
    template <bool FIRST>
    static PORLA_D void mont_round(uint32_t* E, uint32_t* O, const uint32_t* a, uint32_t bi) {
        if (FIRST) {
#pragma unroll
            for (int j = 0; j < 8; j += 2) {
                uint64_t po = (uint64_t)a[j + 1] * bi, pe = (uint64_t)a[j] * bi;
                O[j] = (uint32_t)po;
                O[j + 1] = (uint32_t)(po >> 32);
                E[j] = (uint32_t)pe;
                E[j + 1] = (uint32_t)(pe >> 32);
            }
        } else {
            // E[0] += O[1]; O[j] = a_odd*bi + O[j+2] + carry   (row O moves up by 64 bits)
            asm("add.cc.u32 %0, %0, %2;\n\t"
                "madc.lo.cc.u32 %1, %9, %13, %3;\n\t"
                "madc.hi.cc.u32 %2, %9, %13, %4;\n\t"
                "madc.lo.cc.u32 %3, %10, %13, %5;\n\t"
                "madc.hi.cc.u32 %4, %10, %13, %6;\n\t"
                "madc.lo.cc.u32 %5, %11, %13, %7;\n\t"
                "madc.hi.cc.u32 %6, %11, %13, %8;\n\t"
                "madc.lo.cc.u32 %7, %12, %13, 0;\n\t"
                "madc.hi.u32 %8, %12, %13, 0;"
                : "+r"(E[0]), "+r"(O[0]), "+r"(O[1]), "+r"(O[2]), "+r"(O[3]), "+r"(O[4]),
                  "+r"(O[5]), "+r"(O[6]), "+r"(O[7])
                : "r"(a[1]), "r"(a[3]), "r"(a[5]), "r"(a[7]), "r"(bi));
            // E += a_even*bi ; carry out lands on limb 8 = O[7]
            asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t"
                "madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
                "madc.lo.cc.u32 %2, %10, %13, %2;\n\t"
                "madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
                "madc.lo.cc.u32 %4, %11, %13, %4;\n\t"
                "madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
                "madc.lo.cc.u32 %6, %12, %13, %6;\n\t"
                "madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
                "addc.u32 %8, %8, 0;"
                : "+r"(E[0]), "+r"(E[1]), "+r"(E[2]), "+r"(E[3]), "+r"(E[4]), "+r"(E[5]),
                  "+r"(E[6]), "+r"(E[7]), "+r"(O[7])
                : "r"(a[0]), "r"(a[2]), "r"(a[4]), "r"(a[6]), "r"(bi));
        }
        uint32_t mi = E[0] * P::kInv;
        // O += p_odd * mi  (cannot overflow: O <= T / 2^32 < 2^256)
        asm("mad.lo.cc.u32 %0, %8, %12, %0;\n\t"
            "madc.hi.cc.u32 %1, %8, %12, %1;\n\t"
            "madc.lo.cc.u32 %2, %9, %12, %2;\n\t"
            "madc.hi.cc.u32 %3, %9, %12, %3;\n\t"
            "madc.lo.cc.u32 %4, %10, %12, %4;\n\t"
            "madc.hi.cc.u32 %5, %10, %12, %5;\n\t"
            "madc.lo.cc.u32 %6, %11, %12, %6;\n\t"
            "madc.hi.u32 %7, %11, %12, %7;"
            : "+r"(O[0]), "+r"(O[1]), "+r"(O[2]), "+r"(O[3]), "+r"(O[4]), "+r"(O[5]), "+r"(O[6]),
              "+r"(O[7])
            : "r"(P::mod(1)), "r"(P::mod(3)), "r"(P::mod(5)), "r"(P::mod(7)), "r"(mi));
        // E += p_even * mi ; E[0] becomes 0 ; carry out lands on O[7]
        asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t"
            "madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
            "madc.lo.cc.u32 %2, %10, %13, %2;\n\t"
            "madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
            "madc.lo.cc.u32 %4, %11, %13, %4;\n\t"
            "madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
            "madc.lo.cc.u32 %6, %12, %13, %6;\n\t"
            "madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
            "addc.u32 %8, %8, 0;"
            : "+r"(E[0]), "+r"(E[1]), "+r"(E[2]), "+r"(E[3]), "+r"(E[4]), "+r"(E[5]), "+r"(E[6]),
              "+r"(E[7]), "+r"(O[7])
            : "r"(P::mod(0)), "r"(P::mod(2)), "r"(P::mod(4)), "r"(P::mod(6)), "r"(mi));
    }

    // Montgomery product a*b/2^256 mod p, canonical output, for moduli below 2^254.
    static PORLA_D Fp mul_mont_device(const Fp& a, const Fp& b) {
        uint32_t even[8], odd[8];
        mont_round<true>(even, odd, a.v, b.v[0]);
        mont_round<false>(odd, even, a.v, b.v[1]);
        mont_round<false>(even, odd, a.v, b.v[2]);
        mont_round<false>(odd, even, a.v, b.v[3]);
        mont_round<false>(even, odd, a.v, b.v[4]);
        mont_round<false>(odd, even, a.v, b.v[5]);
        mont_round<false>(even, odd, a.v, b.v[6]);
        mont_round<false>(odd, even, a.v, b.v[7]);
        // T = even + (odd[1..7] one limb lower); T < 2p < 2^255
        Fp r;
        asm("add.cc.u32 %0, %8, %16;\n\t"
            "addc.cc.u32 %1, %9, %17;\n\t"
            "addc.cc.u32 %2, %10, %18;\n\t"
            "addc.cc.u32 %3, %11, %19;\n\t"
            "addc.cc.u32 %4, %12, %20;\n\t"
            "addc.cc.u32 %5, %13, %21;\n\t"
            "addc.cc.u32 %6, %14, %22;\n\t"
            "addc.u32 %7, %15, 0;"
            : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]),
              "=r"(r.v[6]), "=r"(r.v[7])
            : "r"(even[0]), "r"(even[1]), "r"(even[2]), "r"(even[3]), "r"(even[4]), "r"(even[5]),
              "r"(even[6]), "r"(even[7]), "r"(odd[1]), "r"(odd[2]), "r"(odd[3]), "r"(odd[4]),
              "r"(odd[5]), "r"(odd[6]), "r"(odd[7]));
        r.final_sub(0);
        return r;
    }

    // (E, O) += x * s on the two-row layout of mont_round: O (limbs 1..8) takes the odd limbs of x,
    // E (limbs 0..7) the even ones, E's carry-out lands on limb 8 = O[7].
    static PORLA_D void mac_row(uint32_t* E, uint32_t* O, const uint32_t* x, uint32_t s) {
        asm("mad.lo.cc.u32 %0, %8, %12, %0;\n\t"
            "madc.hi.cc.u32 %1, %8, %12, %1;\n\t"
            "madc.lo.cc.u32 %2, %9, %12, %2;\n\t"
            "madc.hi.cc.u32 %3, %9, %12, %3;\n\t"
            "madc.lo.cc.u32 %4, %10, %12, %4;\n\t"
            "madc.hi.cc.u32 %5, %10, %12, %5;\n\t"
            "madc.lo.cc.u32 %6, %11, %12, %6;\n\t"
            "madc.hi.u32 %7, %11, %12, %7;"
            : "+r"(O[0]), "+r"(O[1]), "+r"(O[2]), "+r"(O[3]), "+r"(O[4]), "+r"(O[5]), "+r"(O[6]), "+r"(O[7])
            : "r"(x[1]), "r"(x[3]), "r"(x[5]), "r"(x[7]), "r"(s));
        mac4(E, O[7], x[0], x[2], x[4], x[6], s);
    }

    // Montgomery product-sum (a*b + c*d) / 2^256 mod p with ONE interleaved reduction: each CIOS round
    // adds a*b_i and c*d_i before the reduction step.  Intermediate T < a + c + p < 2^256 and the
    // result is below (2 p^2) / 2^256 + p < 1.5 p, so one conditional subtraction normalises it.
    // Saves one 64-multiply reduction against two separate products (used for y3 in the mixed add).
    static PORLA_D Fp mul2add_mont_device(const Fp& a, const Fp& b, const Fp& c, const Fp& d) {
        uint32_t even[8], odd[8];
        mont_round2<true>(even, odd, a.v, b.v[0], c.v, d.v[0]);
        mont_round2<false>(odd, even, a.v, b.v[1], c.v, d.v[1]);
        mont_round2<false>(even, odd, a.v, b.v[2], c.v, d.v[2]);
        mont_round2<false>(odd, even, a.v, b.v[3], c.v, d.v[3]);
        mont_round2<false>(even, odd, a.v, b.v[4], c.v, d.v[4]);
        mont_round2<false>(odd, even, a.v, b.v[5], c.v, d.v[5]);
        mont_round2<false>(even, odd, a.v, b.v[6], c.v, d.v[6]);
        mont_round2<false>(odd, even, a.v, b.v[7], c.v, d.v[7]);
        Fp r;
        merge_rows(r.v, even, odd);
        r.final_sub(0);
        return r;
    }

    // r = E + (O[1..7] one limb lower): the closing addition of the two-row CIOS
    static PORLA_D void merge_rows(uint32_t* r, const uint32_t* even, const uint32_t* odd) {
        asm("add.cc.u32 %0, %8, %16;\n\t"
            "addc.cc.u32 %1, %9, %17;\n\t"
            "addc.cc.u32 %2, %10, %18;\n\t"
            "addc.cc.u32 %3, %11, %19;\n\t"
            "addc.cc.u32 %4, %12, %20;\n\t"
            "addc.cc.u32 %5, %13, %21;\n\t"
            "addc.cc.u32 %6, %14, %22;\n\t"
            "addc.u32 %7, %15, 0;"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
            : "r"(even[0]), "r"(even[1]), "r"(even[2]), "r"(even[3]), "r"(even[4]), "r"(even[5]),
              "r"(even[6]), "r"(even[7]), "r"(odd[1]), "r"(odd[2]), "r"(odd[3]), "r"(odd[4]),
              "r"(odd[5]), "r"(odd[6]), "r"(odd[7]));
    }

    template <bool FIRST>
    static PORLA_D void mont_round2(uint32_t* E, uint32_t* O, const uint32_t* a, uint32_t bi, const uint32_t* c,
                                    uint32_t di) {
        mont_round_product<FIRST>(E, O, a, bi);
        mac_row(E, O, c, di);
        uint32_t mi = E[0] * P::kInv;
        uint32_t m[8];
#pragma unroll
        for (int j = 0; j < 8; j++) m[j] = P::mod(j);
        mac_row(E, O, m, mi);
    }

    // The product half of a CIOS round (see mont_round): slides the window down one limb and adds a * bi.
    template <bool FIRST>
    static PORLA_D void mont_round_product(uint32_t* E, uint32_t* O, const uint32_t* a, uint32_t bi) {
        if (FIRST) {
#pragma unroll
            for (int j = 0; j < 8; j += 2) {
                uint64_t po = (uint64_t)a[j + 1] * bi, pe = (uint64_t)a[j] * bi;
                O[j] = (uint32_t)po;
                O[j + 1] = (uint32_t)(po >> 32);
                E[j] = (uint32_t)pe;
                E[j + 1] = (uint32_t)(pe >> 32);
            }
        } else {
            asm("add.cc.u32 %0, %0, %2;\n\t"
                "madc.lo.cc.u32 %1, %9, %13, %3;\n\t"
                "madc.hi.cc.u32 %2, %9, %13, %4;\n\t"
                "madc.lo.cc.u32 %3, %10, %13, %5;\n\t"
                "madc.hi.cc.u32 %4, %10, %13, %6;\n\t"
                "madc.lo.cc.u32 %5, %11, %13, %7;\n\t"
                "madc.hi.cc.u32 %6, %11, %13, %8;\n\t"
                "madc.lo.cc.u32 %7, %12, %13, 0;\n\t"
                "madc.hi.u32 %8, %12, %13, 0;"
                : "+r"(E[0]), "+r"(O[0]), "+r"(O[1]), "+r"(O[2]), "+r"(O[3]), "+r"(O[4]),
                  "+r"(O[5]), "+r"(O[6]), "+r"(O[7])
                : "r"(a[1]), "r"(a[3]), "r"(a[5]), "r"(a[7]), "r"(bi));
            mac4(E, O[7], a[0], a[2], a[4], a[6], bi);
        }
    }

    // One round of REDC on the two-row layout without a product term: slide the window down one limb
    // (plain additions), then add mi * p so that the lowest limb cancels.
    template <bool FIRST>
    static PORLA_D void redc_round(uint32_t* E, uint32_t* O) {
        if (!FIRST) {
            // E[0] += O[1]; O[j] = O[j + 2] + carry; the top two limbs of the slid row are zero
            asm("add.cc.u32 %0, %0, %2;\n\t"
                "addc.cc.u32 %1, %3, 0;\n\t"
                "addc.cc.u32 %2, %4, 0;\n\t"
                "addc.cc.u32 %3, %5, 0;\n\t"
                "addc.cc.u32 %4, %6, 0;\n\t"
                "addc.cc.u32 %5, %7, 0;\n\t"
                "addc.cc.u32 %6, %8, 0;\n\t"
                "addc.u32 %7, 0, 0;\n\t"
                "mov.u32 %8, 0;"
                : "+r"(E[0]), "+r"(O[0]), "+r"(O[1]), "+r"(O[2]), "+r"(O[3]), "+r"(O[4]), "+r"(O[5]),
                  "+r"(O[6]), "+r"(O[7]));
        }
        uint32_t m[8];
#pragma unroll
        for (int j = 0; j < 8; j++) m[j] = P::mod(j);
        uint32_t mi = E[0] * P::kInv;
        mac_row(E, O, m, mi);
    }

    // One REDC round with the slide fused into the multiplier's addend operands (no separate additions):
    //   E[0] += O[1];  mi = E[0] * (-1/p);  O[j] = p_odd * mi + O[j + 2] + carry;  E += p_even * mi.
    static PORLA_D void redc_round_fused(uint32_t* E, uint32_t* O) {
        uint32_t mi;
        asm("add.cc.u32 %0, %0, %2;\n\t"
            "mul.lo.u32 %9, %0, %14;\n\t"
            "madc.lo.cc.u32 %1, %10, %9, %3;\n\t"
            "madc.hi.cc.u32 %2, %10, %9, %4;\n\t"
            "madc.lo.cc.u32 %3, %11, %9, %5;\n\t"
            "madc.hi.cc.u32 %4, %11, %9, %6;\n\t"
            "madc.lo.cc.u32 %5, %12, %9, %7;\n\t"
            "madc.hi.cc.u32 %6, %12, %9, %8;\n\t"
            "madc.lo.cc.u32 %7, %13, %9, 0;\n\t"
            "madc.hi.u32 %8, %13, %9, 0;"
            : "+r"(E[0]), "+r"(O[0]), "+r"(O[1]), "+r"(O[2]), "+r"(O[3]), "+r"(O[4]), "+r"(O[5]), "+r"(O[6]),
              "+r"(O[7]), "=&r"(mi)
            : "r"(P::mod(1)), "r"(P::mod(3)), "r"(P::mod(5)), "r"(P::mod(7)), "r"(P::kInv));
        mac4(E, O[7], P::mod(0), P::mod(2), P::mod(4), P::mod(6), mi);
    }

    // REDC of an 8-limb value: lo / 2^256 mod p (result <= p), i.e. the CIOS loop with the multiplier
    // (1, 0, ..., 0).
    static PORLA_D void redc8_device(const uint32_t* lo, uint32_t* r) {
        uint32_t even[8], odd[8];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            even[j] = lo[j];
            odd[j] = 0;
        }
        redc_round<true>(even, odd);
        redc_round_fused(odd, even);
        redc_round_fused(even, odd);
        redc_round_fused(odd, even);
        redc_round_fused(even, odd);
        redc_round_fused(odd, even);
        redc_round_fused(even, odd);
        redc_round_fused(odd, even);
        merge_rows(r, even, odd);
    }

    // a^2 / 2^256 mod p: 36-multiply wide square, REDC of the low half, plus the high half
    // (REDC(lo + hi 2^256) = REDC(lo) + hi; REDC(lo) <= p and hi < p^2 / 2^256 < p / 4).
    static PORLA_D Fp sqr_mont_device(const Fp& a) {
        uint32_t T[16], lo[8];
        sqr_wide_device(a.v, T);
        redc8_device(T, lo);
        Fp r;
        add256(r.v, lo, T + 8);
        r.final_sub(0);
        return r;
    }
#endif

    // portable Montgomery CIOS (host, and reference for the device path)
    PORLA_HD static Fp mul_mont_portable(const Fp& a, const Fp& b) {
        uint32_t t[10];
#pragma unroll
        for (int i = 0; i < 10; i++) t[i] = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            uint64_t c = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                c += (uint64_t)a.v[j] * b.v[i] + t[j];
                t[j] = (uint32_t)c;
                c >>= 32;
            }
            c += t[8];
            t[8] = (uint32_t)c;
            t[9] = (uint32_t)(c >> 32);
            uint32_t m = t[0] * P::kInv;
            c = (uint64_t)m * P::mod(0) + t[0];
            c >>= 32;
#pragma unroll
            for (int j = 1; j < 8; j++) {
                c += (uint64_t)m * P::mod(j) + t[j];
                t[j - 1] = (uint32_t)c;
                c >>= 32;
            }
            c += t[8];
            t[7] = (uint32_t)c;
            t[8] = t[9] + (uint32_t)(c >> 32);
        }
        Fp r;
#pragma unroll
        for (int i = 0; i < 8; i++) r.v[i] = t[i];
        r.final_sub(t[8]);
        return r;
    }

    // portable special-form product for p = 2^256 - C, C = 2^32 + 977 (secp256k1)
    PORLA_HD static Fp mul_special_portable(const Fp& a, const Fp& b) {
        uint32_t t[16];
#pragma unroll
        for (int i = 0; i < 16; i++) t[i] = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            uint64_t c = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                c += (uint64_t)a.v[j] * b.v[i] + t[i + j];
                t[i + j] = (uint32_t)c;
                c >>= 32;
            }
            t[i + 8] = (uint32_t)c;
        }
        // fold 1: r = lo + hi*977 + (hi << 32), 9 limbs + 1 spill bit
        uint32_t r[8];
        uint64_t c = 0;
        uint32_t prev = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            c += (uint64_t)t[8 + i] * 977u + t[i] + prev;
            r[i] = (uint32_t)c;
            c >>= 32;
            prev = t[8 + i];
        }
        c += prev;  // value of limbs 8.. (< 2^34)
        return fold_special_tail(r, c);
    }

    // Folds 2 and 3 of the special-form reduction: r (8 limbs) + c * (2^32 + 977), c < 2^34, then one
    // more wrap if that carried past 2^256, then the conditional subtraction.
    PORLA_HD static Fp fold_special_tail(uint32_t* r, uint64_t c) {
        uint64_t d = (c & 0xffffffffull) * 977u + r[0];
        r[0] = (uint32_t)d;
        d >>= 32;
        d += (c >> 32) * 977u + (c & 0xffffffffull) + r[1];
        r[1] = (uint32_t)d;
        d >>= 32;
        d += (c >> 32) + r[2];
        r[2] = (uint32_t)d;
        d >>= 32;
#pragma unroll
        for (int i = 3; i < 8; i++) {
            d += r[i];
            r[i] = (uint32_t)d;
            d >>= 32;
        }
        // fold 3: a wrap past 2^256 leaves a tiny value; add C once more (cannot wrap again)
        uint64_t e = (uint64_t)r[0] + (d ? 977u : 0u);
        r[0] = (uint32_t)e;
        e >>= 32;
        e += (uint64_t)r[1] + (d ? 1u : 0u);
        r[1] = (uint32_t)e;
        e >>= 32;
#pragma unroll
        for (int i = 2; i < 8; i++) {
            e += r[i];
            r[i] = (uint32_t)e;
            e >>= 32;
        }
        Fp out;
#pragma unroll
        for (int i = 0; i < 8; i++) out.v[i] = r[i];
        out.final_sub(0);
        return out;
    }

#ifdef __CUDA_ARCH__
    // Device special-form reduction of a 16-limb product T for p = 2^256 - (2^32 + 977):
    // fold 1 is  lo + hi * 977 + (hi << 32)  on the two-row layout of mul_wide_device (the even limbs
    // of hi times 977 land on 64-bit aligned slots of `acc`, the odd ones on those of row O, which
    // starts out holding hi itself = the (hi << 32) term); IMAD.WIDE carry chains throughout.
    static PORLA_D Fp fold_special_device(const uint32_t* T) {
        uint32_t acc[10], O[9];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            acc[i] = T[i];
            O[i] = T[8 + i];
        }
        acc[8] = 0;
        O[8] = 0;
        mac4(acc, acc[8], T[8], T[10], T[12], T[14], 977u);
        mac4(O, O[8], T[9], T[11], T[13], T[15], 977u);
        asm("add.cc.u32 %0, %0, %9;\n\t"
            "addc.cc.u32 %1, %1, %10;\n\t"
            "addc.cc.u32 %2, %2, %11;\n\t"
            "addc.cc.u32 %3, %3, %12;\n\t"
            "addc.cc.u32 %4, %4, %13;\n\t"
            "addc.cc.u32 %5, %5, %14;\n\t"
            "addc.cc.u32 %6, %6, %15;\n\t"
            "addc.cc.u32 %7, %7, %16;\n\t"
            "addc.u32 %8, %17, 0;"
            : "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]),
              "+r"(acc[8]), "=r"(acc[9])
            : "r"(O[0]), "r"(O[1]), "r"(O[2]), "r"(O[3]), "r"(O[4]), "r"(O[5]), "r"(O[6]), "r"(O[7]), "r"(O[8]));
        return fold_special_tail(acc, (uint64_t)acc[8] + ((uint64_t)acc[9] << 32));
    }
    static PORLA_D Fp mul_special_device(const Fp& a, const Fp& b) {
        uint32_t T[16];
        mul_wide_device(a.v, b.v, T);
        return fold_special_device(T);
    }
    static PORLA_D Fp sqr_special_device(const Fp& a) {
        uint32_t T[16];
        sqr_wide_device(a.v, T);
        return fold_special_device(T);
    }
#endif

    PORLA_HD friend Fp operator*(const Fp& a, const Fp& b) { return mul(a, b); }
    PORLA_HD Fp sqr() const {
#ifdef __CUDA_ARCH__
        if constexpr (P::kMontgomery && !kCompact) return sqr_mont_device(*this);
        if constexpr (!P::kMontgomery && !kCompact) return sqr_special_device(*this);
#endif
        return mul(*this, *this);
    }
    // a*b + c*d (one reduction on the Montgomery device path)
    PORLA_HD static Fp mul2add(const Fp& a, const Fp& b, const Fp& c, const Fp& d) {
#ifdef __CUDA_ARCH__
        if constexpr (P::kMontgomery && !kCompact) return mul2add_mont_device(a, b, c, d);
#endif
        return mul(a, b) + mul(c, d);
    }

    PORLA_HD static Fp mul_inlined(const Fp& a, const Fp& b) {
        if (P::kMontgomery) {
#ifdef __CUDA_ARCH__
            return mul_mont_device(a, b);
#else
            return mul_mont_portable(a, b);
#endif
        } else {
#ifdef __CUDA_ARCH__
            return mul_special_device(a, b);
#else
            return mul_special_portable(a, b);
#endif
        }
    }
    PORLA_HD static Fp mul(const Fp& a, const Fp& b) {
#ifdef __CUDA_ARCH__
        if constexpr (kCompact) return fp_mul_outlined<P>(a, b);
#endif
        return mul_inlined(a, b);
    }

    // to/from the internal representation (Montgomery for BN254, identity for secp256k1)
    PORLA_HD Fp to_internal() const {
        if (!P::kMontgomery) return *this;
        Fp r2;
#pragma unroll
        for (int i = 0; i < 8; i++) r2.v[i] = P::r2(i);
        return mul(*this, r2);
    }
    PORLA_HD Fp from_internal() const {
        if (!P::kMontgomery) return *this;
        Fp o = zero();
        o.v[0] = 1;
        return mul(*this, o);
    }

    // a^(p-2) by square-and-multiply: ~380 products on the multiplier pipe, a dependent chain (272 k cycles on a lone warp).
    // Kept as the reference the binary-GCD routine is tested against.
    PORLA_HD Fp inverse_fermat() const {
        uint32_t e[8];
#pragma unroll
        for (int i = 0; i < 8; i++) e[i] = P::mod(i);
        e[0] -= 2;  // both moduli end in ...47 / ...2f: no borrow
        Fp r = one();
        for (int i = 255; i >= 0; i--) {
            r = r.sqr();
            if ((e[i >> 5] >> (i & 31)) & 1u) r = mul(r, *this);
        }
        return r;
    }

    // Inverse in the field's internal form by the binary GCD of fp_inv.cuh (77 k cycles on a lone warp, mostly plain ALU
    // work).  For the Montgomery representative a R the plain inverse is a^-1 R^-1; two Montgomery products with R^2 lift
    // it to a^-1 R.  The inverse of zero is zero, as with the Fermat routine.
    PORLA_HD Fp inverse() const {
        Fp r;
#ifdef __CUDA_ARCH__
        fp_inverse_plain_outlined<P>(v, r.v);
#else
        fp_inverse_plain<P, P::kBits>(v, r.v);
#endif
        if (P::kMontgomery) {
            Fp r2;
#pragma unroll
            for (int i = 0; i < 8; i++) r2.v[i] = P::r2(i);
            r = mul(mul(r, r2), r2);
        }
        return r;
    }
};

#ifdef __CUDACC__
template <class P>
__device__ __noinline__ Fp<P, true> fp_mul_outlined(Fp<P, true> a, Fp<P, true> b) {
    return Fp<P, true>::mul_inlined(a, b);
}
#endif

}  // namespace porla
