// Short-Weierstrass group law for a = 0 curves (BN254 G1: y^2 = x^3 + 3, secp256k1: y^2 = x^3 + 7)
// in extended-Jacobian "XYZZ" coordinates (x = X/ZZ, y = Y/ZZZ, ZZ^3 = ZZZ^2).
//
// This is the coordinate system gnark-crypto's MultiExp keeps its buckets in (SURVEY.md
// Appendix B) and replaces secp256k1's Jacobian gej_add_ge_var
// (/root/reference/porla/Utils/secp256k1_lib/group_impl.h:389) as the bucket update.
// All routines handle the exceptional cases (infinity, P + P, P - P) exactly, because Porla's
// inputs contain them (alignment MACs start as infinity, Server.hpp:1534-1535) and parity is
// judged on canonical affine bytes.
#pragma once
#include "fp.cuh"

namespace porla {

template <class F>
struct alignas(16) Affine {
    F x, y;  // infinity is encoded as x = y = 0 (not on either curve)
    PORLA_HD bool is_inf() const { return x.is_zero() && y.is_zero(); }
    PORLA_HD static Affine inf() { return Affine{F::zero(), F::zero()}; }
    PORLA_HD Affine neg() const { return Affine{x, y.neg()}; }
};

template <class F>
struct alignas(16) XYZZ {
    F x, y, zz, zzz;

    PORLA_HD bool is_inf() const { return zz.is_zero(); }
    PORLA_HD static XYZZ inf() { return XYZZ{F::zero(), F::zero(), F::zero(), F::zero()}; }
    PORLA_HD static XYZZ from_affine(const Affine<F>& p) {
        if (p.is_inf()) return inf();
        return XYZZ{p.x, p.y, F::one(), F::one()};
    }
    PORLA_HD XYZZ neg() const { return XYZZ{x, y.neg(), zz, zzz}; }

    // 2 * (affine p), p finite.  mdbl-2008-s-1 with a = 0.
    PORLA_HD static XYZZ dbl_affine(const Affine<F>& p) {
        if (p.y.is_zero()) return inf();  // order-2 point: cannot occur on prime-order curves
        F u = p.y.dbl();
        F v = u.sqr();
        F w = u * v;
        F s = p.x * v;
        F xx = p.x.sqr();
        F m = xx.dbl() + xx;
        XYZZ r;
        r.x = m.sqr() - s.dbl();
        r.y = m * (s - r.x) - w * p.y;
        r.zz = v;
        r.zzz = w;
        return r;
    }

    // 2 * this.  dbl-2008-s-1 with a = 0.
    PORLA_HD XYZZ dbl() const {
        if (is_inf()) return *this;
        F u = y.dbl();
        F v = u.sqr();
        F w = u * v;
        F s = x * v;
        F xx = x.sqr();
        F m = xx.dbl() + xx;
        XYZZ r;
        r.x = m.sqr() - s.dbl();
        r.y = m * (s - r.x) - w * y;
        r.zz = v * zz;
        r.zzz = w * zzz;
        return r;
    }

    // this += affine q.  madd-2008-s: 8M + 2S on the generic path.
    PORLA_HD void madd(const Affine<F>& q) {
        if (q.is_inf()) return;
        if (is_inf()) {
            *this = XYZZ{q.x, q.y, F::one(), F::one()};
            return;
        }
        madd_finite(q);
    }

    // this += affine q where neither operand is infinity (the bucket-accumulation hot op).
    PORLA_HD void madd_finite(const Affine<F>& q) {
        F p = q.x * zz - x;
        F r = q.y * zzz - y;
        if (p.is_zero()) {
            if (r.is_zero()) *this = dbl_affine(q);
            else *this = inf();
            return;
        }
        F pp = p.sqr();
        F ppp = p * pp;
        F qq = x * pp;
        F x3 = r.sqr() - ppp - qq.dbl();
        y = F::mul2add(r, qq - x3, y.neg(), ppp);   // r (qq - x3) - y ppp with one reduction
        x = x3;
        zz = zz * pp;
        zzz = zzz * ppp;
    }

    // this += o.  add-2008-s: 12M + 2S on the generic path.
    PORLA_HD void add(const XYZZ& o) {
        if (o.is_inf()) return;
        if (is_inf()) {
            *this = o;
            return;
        }
        F u1 = x * o.zz;
        F u2 = o.x * zz;
        F s1 = y * o.zzz;
        F s2 = o.y * zzz;
        F p = u2 - u1;
        F r = s2 - s1;
        if (p.is_zero()) {
            if (r.is_zero()) *this = dbl();
            else *this = inf();
            return;
        }
        F pp = p.sqr();
        F ppp = p * pp;
        F qq = u1 * pp;
        F x3 = r.sqr() - ppp - qq.dbl();
        y = r * (qq - x3) - s1 * ppp;
        x = x3;
        zz = zz * o.zz * pp;
        zzz = zzz * o.zzz * ppp;
    }

    // canonical affine form: one field inversion.  1/ZZ = (ZZ / ZZZ)^2 because ZZ^3 = ZZZ^2.
    PORLA_HD Affine<F> to_affine() const {
        if (is_inf()) return Affine<F>::inf();
        F i3 = zzz.inverse();
        F t = zz * i3;
        Affine<F> a;
        a.x = x * t.sqr();
        a.y = y * i3;
        return a;
    }
};

// k * p for a small non-negative k (used by the bucket reduction to weight a chunk sum)
template <class F>
PORLA_HD XYZZ<F> mul_small(const XYZZ<F>& p, uint32_t k) {
    XYZZ<F> r = XYZZ<F>::inf();
    if (k == 0 || p.is_inf()) return r;
    int top = 31;
    while (!((k >> top) & 1u)) top--;
    for (int i = top; i >= 0; i--) {
        r = r.dbl();
        if ((k >> i) & 1u) r.add(p);
    }
    return r;
}

// Curve tags ------------------------------------------------------------------------------
using Bn254Fp = Fp<Bn254FpParams>;
using SecpFp = Fp<Secp256k1FpParams>;
using Bn254FpCompact = Fp<Bn254FpParams, true>;
using SecpFpCompact = Fp<Secp256k1FpParams, true>;

struct Bn254 {
    using F = Bn254Fp;
    using FC = Bn254FpCompact;  // same layout, non-inlined multiplier (cold kernels)
    static constexpr int kFieldBits = 254;      // bit length of the base-field modulus
    static constexpr int kScalarBits = 254;     // bits the window recoder covers (r < 2^254)
    static constexpr bool kHalveScalar = false;
    // GLV: phi(x, y) = (beta x, y) = lambda (x, y) with beta^3 = 1 in Fp, lambda^3 = 1 mod r.  A scalar k splits as
    // k = k1 + k2 lambda with |k1|, |k2| < 2^127 (lattice basis (a1, b1), (a2, b2), a1 b2 - a2 b1 = r; constants
    // re-derived independently and compared limb by limb in tests/test_oracle.py), so an n-term MSM becomes a
    // 2n-term MSM over (P_i, phi(P_i)) with half as many windows, i.e. half as many buckets to reduce.
    static constexpr bool kGlv = true;
    static constexpr int kGlvBits = 127;
    // bucket count up to which the bucket reduction runs on quads (k_reduce_scan): measured crossover against k_reduce
    // (0.93 against 0.92 ms at 983 k buckets, 0.66 against 0.71 ms for one set of 524 k)
    static constexpr uint32_t kReduceQuadMax = 600000;
    // butterfly count up to which a stage of the FFT in the exponent runs on quads (k_butterfly_quad): at most two warps of
    // quads per scheduler, 148 x 4 x 2 x 8
    static constexpr uint32_t kButterflyQuadMax = 9472;
    PORLA_HD static constexpr uint32_t glv_beta_mont(int i) {   // beta * 2^256 mod p
        constexpr uint32_t m[8] = {0xd782e155u, 0x71930c11u, 0xffbe3323u, 0xa6bb947cu,
                                   0xd4741444u, 0xaa303344u, 0x26594943u, 0x2c3b3f0du};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t glv_g1(int i) {   // floor(2^256 * b2 / r)
        constexpr uint32_t m[3] = {0xc7e0b3d7u, 0xd91d232eu, 0x2u};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t glv_g2(int i) {   // floor(2^256 * (-b1) / r)
        constexpr uint32_t m[5] = {0x391eb18du, 0x7a7bd9d4u, 0xa773d2cfu, 0x4ccef014u, 0x2u};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t glv_a1(int i) {   // a1 = b2
        constexpr uint32_t m[2] = {0x94d213e3u, 0x89d32568u};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t glv_a2(int i) {
        constexpr uint32_t m[4] = {0x1221250bu, 0x0be4e154u, 0xeeb859fdu, 0x6f4d8248u};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t glv_nb1(int i) {  // -b1
        constexpr uint32_t m[4] = {0x7d4f1128u, 0x8211bbebu, 0xeeb859fcu, 0x6f4d8248u};
        return m[i];
    }
    // r (scalar field order), little-endian 32-bit limbs
    PORLA_HD static constexpr uint32_t order(int i) {
        constexpr uint32_t m[8] = {0xf0000001u, 0x43e1f593u, 0x79b97091u, 0x2833e848u,
                                   0x8181585du, 0xb85045b6u, 0xe131a029u, 0x30644e72u};
        return m[i];
    }
    static constexpr uint32_t kB = 3;
};

struct Secp256k1 {
    using F = SecpFp;
    using FC = SecpFpCompact;
    // n is just below 2^256: scalars above n/2 are recoded as -(n - s), so 255 magnitude bits (plus the
    // carry of the signed digits) span exactly 16 windows of 16 bits instead of 17 with a 1-bit top window.
    static constexpr int kFieldBits = 256;
    static constexpr int kScalarBits = 255;
    static constexpr bool kHalveScalar = true;
    // no GLV in the MSM: the split halves of a secp256k1 scalar reach 2^128 (they need 129 bits with the signed digits'
    // carry), so 2n terms x 9 windows of 16 bits would cost more bucket updates than n terms x 16 windows
    static constexpr bool kGlv = false;
    static constexpr int kGlvBits = 0;
    // quads up to 300 k buckets (the cheaper special-form product moves the crossover: at 524 k buckets, 2^18 / 2^20 terms,
    // k_reduce 1.231 / 2.880 ms per MSM against 1.254 / 2.904 ms on quads; 2^16: quads 0.63 against 0.70 ms)
    static constexpr uint32_t kReduceQuadMax = 300000;
    // quads up to 9472 butterflies as for BN254: quad 0.41 / 0.54 / 1.07 ms per stage at 4096 / 8192 / 16384 butterflies
    // against 0.91 / 0.93 / 0.99 ms for k_butterfly (one B200, 1000 W; profiles/r04_secp_butterfly_times.txt)
    static constexpr uint32_t kButterflyQuadMax = 9472;
    // The butterflies of the FFT in the exponent use the endomorphism all the same: phi(x, y) = (beta x, y) = lambda (x, y),
    // k = k1 + k2 lambda with |k1|, |k2| < 2^128 (glv_split_secp256k1 below).  Only k_butterfly(_quad) and the host
    // butterfly read these constants; kGlv above keeps tables, plan codes and MSMs free of the split.
    PORLA_HD static constexpr uint32_t glv_beta_mont(int i) {   // beta in internal form, which is plain for this field
        constexpr uint32_t m[8] = {0x719501eeu, 0xc1396c28u, 0x12f58995u, 0x9cf04975u,
                                   0xac3434e9u, 0x6e64479eu, 0x657c0710u, 0x7ae96a2bu};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t glv_lambda(int i) {
        constexpr uint32_t m[8] = {0x1b23bd72u, 0xdf02967cu, 0x20816678u, 0x122e22eau,
                                   0x8812645au, 0xa5261c02u, 0xc05c30e0u, 0x5363ad4cu};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t glv_g1(int i) {   // round(2^384 * b2 / n)
        constexpr uint32_t m[8] = {0x45dbb031u, 0xe893209au, 0x71e8ca7fu, 0x3daa8a14u,
                                   0x9284eb15u, 0xe86c90e4u, 0xa7d46bcdu, 0x3086d221u};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t glv_g2(int i) {   // round(2^384 * (-b1) / n)
        constexpr uint32_t m[8] = {0x8ac47f71u, 0x1571b4aeu, 0x9df506c6u, 0x221208acu,
                                   0x0abfe4c4u, 0x6f547fa9u, 0x010e8828u, 0xe4437ed6u};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t glv_a1(int i) {   // a1 = b2
        constexpr uint32_t m[4] = {0x9284eb15u, 0xe86c90e4u, 0xa7d46bcdu, 0x3086d221u};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t glv_a2(int i) {
        constexpr uint32_t m[5] = {0x9d44cfd8u, 0x57c1108du, 0xa8e2f3f6u, 0x14ca50f7u, 0x00000001u};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t glv_nb1(int i) {  // -b1
        constexpr uint32_t m[4] = {0x0abfe4c3u, 0x6f547fa9u, 0x010e8828u, 0xe4437ed6u};
        return m[i];
    }
    PORLA_HD static constexpr uint32_t order(int i) {
        constexpr uint32_t m[8] = {0xd0364141u, 0xbfd25e8cu, 0xaf48a03bu, 0xbaaedce6u,
                                   0xfffffffeu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
        return m[i];
    }
    static constexpr uint32_t kB = 7;
};

// out = a * b mod 2^(32*NO) on 32-bit limbs (schoolbook; a few dozen IMADs per scalar)
template <int NA, int NB, int NO>
PORLA_HD void mul_limbs(const uint32_t* a, const uint32_t* b, uint32_t* out) {
#pragma unroll
    for (int i = 0; i < NO; i++) out[i] = 0;
#pragma unroll
    for (int i = 0; i < NA; i++) {
        uint64_t carry = 0;
#pragma unroll
        for (int j = 0; j < NB; j++) {
            if (i + j < NO) {
                uint64_t v = (uint64_t)a[i] * b[j] + out[i + j] + carry;
                out[i + j] = (uint32_t)v;
                carry = v >> 32;
            }
        }
        if (i + NB < NO) out[i + NB] = (uint32_t)carry;
    }
}

// k (reduced mod n) -> |k1|, |k2| < 2^128 and their signs, k = k1 + k2 * lambda (mod n); host and device.
//   c1 = round(k * g1 / 2^384),  c2 = round(k * g2 / 2^384)     (libsecp256k1's secp256k1_scalar_split_lambda)
//   k1 = k - c1 a1 - c2 a2,  k2 = c1 (-b1) - c2 a1               (exact, evaluated mod 2^192 in two's complement)
// The roundings matter: floors (as BN254's glv_split takes them) leave 129-bit halves, one digit more than the 64 two-bit
// digits of k_butterfly_quad.  Bound checked on corner scalars and 2 * 10^5 random ones in tests/test_secp_butterfly.py.
PORLA_HD void glv_split_secp256k1(const uint32_t* k, uint32_t* k1, uint32_t* k2, uint32_t& neg1, uint32_t& neg2) {
    using C = Secp256k1;
    uint32_t g1[8], g2[8], a1[4], a2[5], nb1[4];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        g1[i] = C::glv_g1(i);
        g2[i] = C::glv_g2(i);
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        a1[i] = C::glv_a1(i);
        nb1[i] = C::glv_nb1(i);
    }
#pragma unroll
    for (int i = 0; i < 5; i++) a2[i] = C::glv_a2(i);
    uint32_t t1[16], t2[16];
    mul_limbs<8, 8, 16>(k, g1, t1);
    mul_limbs<8, 8, 16>(k, g2, t2);
    uint32_t c1[4], c2[4];   // bits 384.. plus bit 383 (both below 2^128 after the rounding)
    uint32_t r1 = t1[11] >> 31, r2 = t2[11] >> 31;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        uint64_t x = (uint64_t)t1[12 + i] + r1;
        c1[i] = (uint32_t)x;
        r1 = (uint32_t)(x >> 32);
        uint64_t y = (uint64_t)t2[12 + i] + r2;
        c2[i] = (uint32_t)y;
        r2 = (uint32_t)(y >> 32);
    }
    uint32_t p1[6], p2[6], q1[6], q2[6];
    mul_limbs<4, 4, 6>(c1, a1, p1);
    mul_limbs<4, 5, 6>(c2, a2, p2);
    mul_limbs<4, 4, 6>(c1, nb1, q1);
    mul_limbs<4, 4, 6>(c2, a1, q2);   // b2 = a1
    uint32_t v1[6], v2[6];
    uint32_t borrow = 0, borrow2 = 0, borrow3 = 0;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        uint64_t d = (uint64_t)k[i] - p1[i] - borrow;
        borrow = (uint32_t)(d >> 63);
        uint64_t e = (uint64_t)(uint32_t)d - p2[i] - borrow2;
        borrow2 = (uint32_t)(e >> 63);
        v1[i] = (uint32_t)e;
        uint64_t f = (uint64_t)q1[i] - q2[i] - borrow3;
        borrow3 = (uint32_t)(f >> 63);
        v2[i] = (uint32_t)f;
    }
    neg1 = v1[5] >> 31;
    neg2 = v2[5] >> 31;
    uint32_t cy1 = neg1, cy2 = neg2;   // two's complement negation where negative
#pragma unroll
    for (int i = 0; i < 6; i++) {
        uint64_t x = (uint64_t)(neg1 ? ~v1[i] : v1[i]) + cy1;
        v1[i] = (uint32_t)x;
        cy1 = (uint32_t)(x >> 32);
        uint64_t y = (uint64_t)(neg2 ? ~v2[i] : v2[i]) + cy2;
        v2[i] = (uint32_t)y;
        cy2 = (uint32_t)(y >> 32);
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        k1[i] = v1[i];
        k2[i] = v2[i];
    }
}

}  // namespace porla
