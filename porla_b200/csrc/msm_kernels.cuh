// Pippenger (bucket-method) multi-scalar multiplication kernels for sm_100a, templated on curve.
//
// Replaces, on the device:
//   * gnark-crypto's G1Affine.MultiExp reached from /root/reference/porla/main.go:136 (and
//     kzg.Commit, main.go:114,164), and
//   * secp256k1_ecmult_pippenger_wnaf, /root/reference/porla/Utils/secp256k1_lib/ecmult_impl.h:492-567.
//
// Pipeline (one or many MSMs per launch sequence; "window slot" = (msm, window)):
//   sort, small / batched    k_digits<COUNT> (signed c-bit recoding of every scalar, histogram of bucket sizes), k_scan_*
//                            (bucket offsets), k_digits<SCATTER> (recode again, one returning atomic per pair)
//   sort, single MSM >= 2^19 k_coarse_count + k_coarse_scan + k_partition_coarse + k_fine_smem (coarse histogram, shared-memory
//                            radix partition, one block per coarse bin sorting it in shared memory; k_big_* for oversized bins),
//                            or the exact histogram + k_partition_coarse + k_partition_fine when a bin cannot fit shared memory
//   k_accumulate             one thread per SLICE of the bucket-sorted pair list: XYZZ += affine, partial sums at the cuts
//   k_stitch, k_stitch_long  the cut buckets' partial sums
//   k_reduce / k_reduce_scan per window slot: sum_k (k+1) B_k by chunked running sums (one thread per chunk) or, up to 600 k
//                            buckets, by suffix scans on quads (four lanes per point, quad.cuh); k_window_sums / k_reduce_top
//   k_finalize               per MSM: Horner over windows, to affine, serialise (single MSMs finish on the host instead)
//   k_butterfly(_quad), k_data_butterfly, k_audit_aggregate, k_align_scalars: the SURVEY 8(f) operations
//
// Data layout in HBM: points are 64-byte affine records (x,y as 8 LE 32-bit limbs in the
// field's internal form, infinity = all zero) read with 128-bit loads; buckets are 128-byte
// XYZZ records; the sorted list is 8 B per (point, window) pair: bucket id, point index | sign.
#pragma once
#include "ec.cuh"
#include "quad.cuh"

namespace porla {

enum ScalarFormat : int { kScalarBE32 = 0, kScalarLE32 = 1 };
enum PointFormat : int { kPointBE64 = 0, kPointLE64 = 1 };

struct MsmShape {
    uint32_t n;          // scalars per MSM
    uint32_t nbatch;     // MSMs in this launch
    uint32_t shared;     // 1: every MSM uses points[0..n), 0: MSM m uses points[m*n .. (m+1)*n)
    int c;               // window bits
    int nwin;            // windows per scalar
    uint32_t nbuckets;   // buckets per window = 2^(c-1)
    uint32_t fixed_n;    // 0: general.  > 0: fixed-base table of stride fixed_n (windows share buckets)
    int glv_wh;          // 0: off.  > 0: GLV, windows per half; nwin = 2 * glv_wh, window w and w + glv_wh share buckets
    uint32_t phi_off;    // GLV: phi(P_i) is the table entry phi_off + i
};

// ---------------------------------------------------------------------------- small helpers
template <class T>
PORLA_D T ld16(const T* p) {  // 16-byte aligned record, 128-bit loads
    T r;
    const uint4* s = reinterpret_cast<const uint4*>(p);
    uint4* d = reinterpret_cast<uint4*>(&r);
#pragma unroll
    for (int i = 0; i < (int)(sizeof(T) / 16); i++) d[i] = __ldg(s + i);
    return r;
}
template <class T>
PORLA_D void st16(T* p, const T& v) {
    uint4* d = reinterpret_cast<uint4*>(p);
    const uint4* s = reinterpret_cast<const uint4*>(&v);
#pragma unroll
    for (int i = 0; i < (int)(sizeof(T) / 16); i++) d[i] = s[i];
}

PORLA_D uint32_t bswap32(uint32_t x) { return __byte_perm(x, 0, 0x0123); }

// 32 bytes -> 8 little-endian limbs
PORLA_D void load_u256(const uint8_t* base, size_t idx, int big_endian, uint32_t* s) {
    const uint4* p = reinterpret_cast<const uint4*>(base + idx * 32);
    uint4 a = __ldg(p), b = __ldg(p + 1);
    if (big_endian) {
        s[7] = bswap32(a.x); s[6] = bswap32(a.y); s[5] = bswap32(a.z); s[4] = bswap32(a.w);
        s[3] = bswap32(b.x); s[2] = bswap32(b.y); s[1] = bswap32(b.z); s[0] = bswap32(b.w);
    } else {
        s[0] = a.x; s[1] = a.y; s[2] = a.z; s[3] = a.w;
        s[4] = b.x; s[5] = b.y; s[6] = b.z; s[7] = b.w;
    }
}
PORLA_D void store_u256(uint8_t* base, size_t idx, int big_endian, const uint32_t* s) {
    uint4* p = reinterpret_cast<uint4*>(base + idx * 32);
    uint4 a, b;
    if (big_endian) {
        a.x = bswap32(s[7]); a.y = bswap32(s[6]); a.z = bswap32(s[5]); a.w = bswap32(s[4]);
        b.x = bswap32(s[3]); b.y = bswap32(s[2]); b.z = bswap32(s[1]); b.w = bswap32(s[0]);
    } else {
        a.x = s[0]; a.y = s[1]; a.z = s[2]; a.w = s[3];
        b.x = s[4]; b.y = s[5]; b.z = s[6]; b.w = s[7];
    }
    p[0] = a;
    p[1] = b;
}

// s mod order (fr.Element.SetBytes semantics, main.go:127; secp256k1: scalars are "not reduced"
// by convert_ZZ_to_scalar, utils.h:180-192, the reference then works mod n).
template <class C>
PORLA_D void reduce_scalar(uint32_t* s) {
    uint32_t m[8], t[8];
#pragma unroll
    for (int i = 0; i < 8; i++) m[i] = C::order(i);
    // 2^256 / r < 6 for BN254, < 2 for secp256k1
    for (int k = 0; k < 6; k++) {
        uint32_t borrow = sub256(t, s, m);
        if (borrow) break;
#pragma unroll
        for (int i = 0; i < 8; i++) s[i] = t[i];
    }
}

// ---------------------------------------------------------------------------- GLV scalar split
// k (reduced mod r) -> |k1|, |k2| < 2^127 and their signs, k = k1 + k2 * lambda (mod r).
//   c1 = floor(k * g1 / 2^256) ~ k b2 / r,  c2 = floor(k * g2 / 2^256) ~ -k b1 / r
//   k1 = k - c1 a1 - c2 a2,  k2 = -c1 b1 - c2 b2        (exact, evaluated mod 2^192 in two's complement)
// Any integers c1, c2 give a valid split; the floors instead of roundings only cost one bit of size
// (bound checked exhaustively on the corners and on 3*10^5 random scalars in tests/test_oracle.py).
template <class C>
PORLA_D void glv_split(const uint32_t* k, uint32_t* k1, uint32_t* k2, uint32_t& neg1, uint32_t& neg2) {
    uint32_t g1[3], g2[5], a1[2], a2[4], nb1[4];
#pragma unroll
    for (int i = 0; i < 3; i++) g1[i] = C::glv_g1(i);
#pragma unroll
    for (int i = 0; i < 5; i++) g2[i] = C::glv_g2(i);
#pragma unroll
    for (int i = 0; i < 2; i++) a1[i] = C::glv_a1(i);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        a2[i] = C::glv_a2(i);
        nb1[i] = C::glv_nb1(i);
    }
    uint32_t t1[11], t2[13];
    mul_limbs<8, 3, 11>(k, g1, t1);
    mul_limbs<8, 5, 13>(k, g2, t2);
    const uint32_t* c1 = t1 + 8;   // 2 limbs (c1 < 2^64)
    const uint32_t* c2 = t2 + 8;   // 4 limbs (c2 < 2^127)
    uint32_t p1[6], p2[6], q1[6], q2[6];
    mul_limbs<2, 2, 6>(c1, a1, p1);
    mul_limbs<4, 4, 6>(c2, a2, p2);
    mul_limbs<2, 4, 6>(c1, nb1, q1);
    mul_limbs<4, 2, 6>(c2, a1, q2);   // b2 = a1
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

// secp256k1: its own routine (rounded c1, c2 and its limb sizes: ec.cuh), shared with the host butterfly
template <>
PORLA_D void glv_split<Secp256k1>(const uint32_t* k, uint32_t* k1, uint32_t* k2, uint32_t& neg1, uint32_t& neg2) {
    glv_split_secp256k1(k, k1, k2, neg1, neg2);
}

// ---------------------------------------------------------------------------- scalar preparation
// scalar idx -> canonical magnitude (reduced mod the order; secp256k1: min(s, n - s) with flip = 1 when negated)
template <class C>
PORLA_D uint32_t canonical_scalar(const uint8_t* __restrict__ scalars, size_t idx, int big_endian, uint32_t* s) {
    load_u256(scalars, idx, big_endian, s);
    reduce_scalar<C>(s);
    uint32_t flip = 0;
    if (C::kHalveScalar) {
        uint32_t ord[8], t[8], u[8];
#pragma unroll
        for (int k = 0; k < 8; k++) ord[k] = C::order(k);
        sub256(t, ord, s);                 // order - s  (s < order)
        if (sub256(u, t, s)) {             // order - s < s
            flip = 1;
#pragma unroll
            for (int k = 0; k < 8; k++) s[k] = t[k];
        }
    }
    return flip;
}

// scalar idx, reduced mod r and GLV-split -> |k1|, |k2| (4 limbs each) and their signs (neg = 1: negate the point)
template <class C>
PORLA_D void glv_scalar(const uint8_t* __restrict__ scalars, size_t idx, int big_endian, uint32_t* k1, uint32_t* k2,
                        uint32_t& neg1, uint32_t& neg2) {
    uint32_t k[8];
    load_u256(scalars, idx, big_endian, k);
    reduce_scalar<C>(k);
    glv_split<C>(k, k1, k2, neg1, neg2);
}

// out[i] = beta * x_i: the x coordinate of the endomorphism image (beta x_i, y_i) of every table entry
template <class C>
__global__ void __launch_bounds__(128)
k_phi_table(const Affine<typename C::F>* __restrict__ in, uint32_t n, typename C::F* __restrict__ out) {
    using F = typename C::F;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Affine<F> p;
    {   // plain loads: `in` may have been written earlier on this stream by the butterfly kernel
        const uint4* s = reinterpret_cast<const uint4*>(in + i);
        uint4* d = reinterpret_cast<uint4*>(&p);
#pragma unroll
        for (int q = 0; q < 4; q++) d[q] = s[q];
    }
    F beta;
#pragma unroll
    for (int q = 0; q < 8; q++) beta.v[q] = C::glv_beta_mont(q);
    st16(out + i, p.x * beta);      // infinity (0, 0) stays (0, 0)
}

// ---------------------------------------------------------------------------- import / export
// External bytes -> internal affine records.  BN254: gnark Marshal layout X||Y big-endian with
// the two flag bits of byte 0 masked (fp.Element.SetBytes reduces mod p); 64 zero bytes is
// infinity.  flags[i] = 1 marks infinity so the recoder can drop the pair.
template <class C>
__global__ void k_import_points(const uint8_t* __restrict__ in, int fmt, int mask_top2, uint32_t n,
                                Affine<typename C::F>* __restrict__ out, uint8_t* __restrict__ flags,
                                uint32_t* __restrict__ inf_count) {
    using F = typename C::F;
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    F x, y;
    load_u256(in, 2 * (size_t)i, fmt == kPointBE64, x.v);
    load_u256(in, 2 * (size_t)i + 1, fmt == kPointBE64, y.v);
    // gnark G1Affine.SetBytes: the top two bits of byte 0 select the encoding
    //   00 uncompressed X||Y, 01 compressed infinity, 10/11 compressed (y smallest/largest)
    uint32_t flag = mask_top2 ? (x.v[7] >> 30) : 0u;
    if (mask_top2) x.v[7] &= 0x3fffffffu;
    uint32_t m[8];
#pragma unroll
    for (int j = 0; j < 8; j++) m[j] = F::Params::mod(j);
    // reduce below p (inputs are < 2^256; p > 2^253 so a few subtractions suffice)
    for (int k = 0; k < 6; k++) {
        F t;
        if (sub256(t.v, x.v, m)) break;
        x = t;
    }
    for (int k = 0; k < 6; k++) {
        F t;
        if (sub256(t.v, y.v, m)) break;
        y = t;
    }
    if (flag == 1u) {
        x = F::zero();
        y = F::zero();
    } else if (flag >= 2u) {
        // compressed point (never produced by Porla for MSM inputs; handled for SetBytes parity):
        // y = sqrt(x^3 + b) = (x^3 + b)^((p+1)/4), p = 3 mod 4; pick the root by the flag
        F xi = x.to_internal();
        F bb = F::zero();
        bb.v[0] = C::kB;
        F rhs = xi.sqr() * xi + bb.to_internal();
        uint32_t e[8], one[8] = {1, 0, 0, 0, 0, 0, 0, 0};
        add256(e, m, one);
#pragma unroll
        for (int j = 0; j < 8; j++) e[j] = (e[j] >> 2) | (j < 7 ? (e[j + 1] << 30) : 0u);
        F r = F::one();
        for (int b = 255; b >= 0; b--) {
            r = r.sqr();
            if ((e[b >> 5] >> (b & 31)) & 1u) r = r * rhs;
        }
        if (r.sqr() != rhs) {
            x = F::zero();
            y = F::zero();
        } else {
            F yc = r.from_internal();
            uint32_t half[8], t[8];
#pragma unroll
            for (int j = 0; j < 8; j++) half[j] = (m[j] >> 1) | (j < 7 ? (m[j + 1] << 31) : 0u);
            bool largest = sub256(t, half, yc.v) != 0;  // y > (p-1)/2
            if (largest != (flag == 3u)) sub256(yc.v, m, yc.v);
            y = yc;
        }
    }
    bool inf = x.is_zero() && y.is_zero();
    Affine<F> p{x.to_internal(), y.to_internal()};
    st16(out + i, p);
    if (flags) flags[i] = inf ? 1 : 0;
    if (inf && inf_count) atomicAdd(inf_count, 1u);
}

// Jacobian points (IPA-mode MACs, secp256k1_gej) -> internal affine records and their flags: x = X / Z^2, y = Y / Z^3 with
// one inversion per point, skipped when Z = 1 (every point this library returns).  xyz: canonical X, Y, Z, 8 LE limbs
// each; inf: the gej's infinity flag.
template <class C>
__global__ void __launch_bounds__(128)
k_import_jacobian(const uint32_t* __restrict__ xyz, const uint8_t* __restrict__ inf, uint32_t n,
                  Affine<typename C::F>* __restrict__ out, uint8_t* __restrict__ flags) {
    using F = typename C::F;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    F x, y, z;
#pragma unroll
    for (int q = 0; q < 8; q++) {
        x.v[q] = xyz[24 * (size_t)i + q];
        y.v[q] = xyz[24 * (size_t)i + 8 + q];
        z.v[q] = xyz[24 * (size_t)i + 16 + q];
    }
    x = x.to_internal();
    y = y.to_internal();
    z = z.to_internal();
    Affine<F> p = Affine<F>::inf();
    if (!inf[i] && !z.is_zero()) {
        const F zi = z == F::one() ? z : z.inverse(), zi2 = zi.sqr();
        p.x = x * zi2;
        p.y = y * zi2 * zi;
    }
    st16(out + i, p);
    flags[i] = p.is_inf() ? 1 : 0;
}

// internal affine -> external bytes (inverse of the above)
template <class C>
__global__ void k_export_points(const Affine<typename C::F>* __restrict__ in, uint32_t n, int fmt,
                                uint8_t* __restrict__ out) {
    using F = typename C::F;
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Affine<F> p = ld16(in + i);
    F x = p.x.from_internal(), y = p.y.from_internal();
    store_u256(out, 2 * (size_t)i, fmt == kPointBE64, x.v);
    store_u256(out, 2 * (size_t)i + 1, fmt == kPointBE64, y.v);
}

// Fixed-base expansion: out[w*n + i] = 2^(c*w) * P_i, affine, for w < nwin (out[i] = P_i).
template <class C>
__global__ void __launch_bounds__(128)
k_precompute_windows(const Affine<typename C::FC>* __restrict__ in, uint32_t n, int c, int nwin,
                     Affine<typename C::FC>* __restrict__ out) {
    using F = typename C::FC;
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Affine<F> p = ld16(in + i);
    st16(out + i, p);
    XYZZ<F> r = XYZZ<F>::from_affine(p);
    for (int w = 1; w < nwin; w++) {
        for (int k = 0; k < c; k++) r = r.dbl();
        Affine<F> a = r.to_affine();
        st16(out + (size_t)w * n + i, a);
        r = XYZZ<F>::from_affine(a);   // restart from the affine form: keeps zz = zzz = 1
    }
}

// ---------------------------------------------------------------------------- recoding
// Signed c-bit digits: d_w in [-2^(c-1), 2^(c-1)], bucket id |d_w| - 1; nwin*c > bits of the
// order, so the top digit never overflows.
template <class C, bool SCATTER, bool GLV>
__global__ void __launch_bounds__(256)
k_digits(const uint8_t* __restrict__ scalars, int big_endian,
         const uint8_t* __restrict__ inf_flags, MsmShape sh, int w_begin, int w_end,
         uint32_t* __restrict__ counters, uint2* __restrict__ sorted) {
    // Only windows [w_begin, w_end) are emitted: the host scatters a few windows per launch so that
    // the region of `sorted` being written (n * 8 B per window) stays L2-resident and the 8-byte
    // stores merge into full sectors before they reach HBM.
    const uint64_t total = (uint64_t)sh.n * sh.nbatch;
    const uint32_t half = 1u << (sh.c - 1);
    const uint32_t mask = (1u << sh.c) - 1u;
    constexpr int kBatch = 8;  // independent atomics kept in flight per thread
    // limbs of the value being recoded: the scalar (s[8] = 0), or with GLV the two halves |k1| in s[0..3],
    // |k2| in s[5..8] (s[4] = s[9] = 0), window w >= glv_wh reading the second half
    constexpr int kLimbs = GLV ? 10 : 9;
    const int wh = GLV ? sh.glv_wh : sh.nwin;
    for (uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t m = (uint32_t)(idx / sh.n);
        uint32_t i = (uint32_t)(idx - (uint64_t)m * sh.n);
        uint32_t pidx = sh.shared ? i : (uint32_t)idx;
        if (inf_flags && inf_flags[pidx]) continue;
        uint32_t s[kLimbs];
        uint32_t flip[2] = {0, 0};   // negate the point (per half with GLV)
        if constexpr (GLV) {
            glv_scalar<C>(scalars, idx, big_endian, s, s + 5, flip[0], flip[1]);
            s[4] = 0;
            s[9] = 0;
        } else {
            s[8] = 0;
            flip[0] = canonical_scalar<C>(scalars, idx, big_endian, s);
        }
        uint32_t carry = 0;
        // general: one bucket set per (msm, window); fixed-base: one per msm, the window selects the
        // pre-multiplied copy 2^(c*w) * P_i of the point instead; GLV: one per (msm, window of a half)
        const uint32_t slot_base = sh.fixed_n ? m * sh.nbuckets : m * (uint32_t)wh * sh.nbuckets;
        for (int w0 = 0; w0 < w_end; w0 += kBatch) {
            uint32_t bucket[kBatch], val[kBatch];
#pragma unroll
            for (int k = 0; k < kBatch; k++) {
                int w = w0 + k;
                bucket[k] = 0xffffffffu;
                val[k] = 0;
                if (w < sh.nwin) {
                    const int h = GLV && w >= wh ? 1 : 0;
                    const int wl = w - h * wh;
                    if (GLV && wl == 0) carry = 0;
                    uint32_t pos = (uint32_t)wl * sh.c + (GLV ? 160u * h : 0u);
                    uint32_t word = pos >> 5, sft = pos & 31;
                    uint32_t lo = s[word < kLimbs - 1 ? word : kLimbs - 1];
                    uint32_t hi = s[word < kLimbs - 2 ? word + 1 : kLimbs - 1];
                    uint32_t d = (__funnelshift_r(lo, hi, sft) & mask) + carry;
                    uint32_t dneg = d > half;
                    carry = dneg;
                    uint32_t mag = dneg ? ((1u << sh.c) - d) : d;
                    uint32_t neg = dneg ^ flip[h];
                    if (mag != 0 && w >= w_begin && w < w_end) {
                        if (sh.fixed_n) {
                            bucket[k] = slot_base + (mag - 1);
                            val[k] = ((uint32_t)w * sh.fixed_n + pidx) | (neg << 31);
                        } else {
                            bucket[k] = slot_base + (uint32_t)wl * sh.nbuckets + (mag - 1);
                            val[k] = (pidx + (h ? sh.phi_off : 0u)) | (neg << 31);
                        }
                    }
                }
            }
            if (!SCATTER) {
#pragma unroll
                for (int k = 0; k < kBatch; k++)
                    if (bucket[k] != 0xffffffffu) atomicAdd(counters + bucket[k], 1u);
            } else {
                uint32_t at[kBatch];
#pragma unroll
                for (int k = 0; k < kBatch; k++)
                    at[k] = bucket[k] != 0xffffffffu ? atomicAdd(counters + bucket[k], 1u) : 0u;
#pragma unroll
                for (int k = 0; k < kBatch; k++)
                    if (bucket[k] != 0xffffffffu) sorted[at[k]] = make_uint2(bucket[k], val[k]);
            }
        }
    }
}

// ---------------------------------------------------------------------------- prefix sum
constexpr int kScanThreads = 512;
constexpr int kScanItems = 4;
constexpr int kScanTile = kScanThreads * kScanItems;

// block-wide exclusive scan of one value per thread; returns the exclusive prefix, total in *sum
PORLA_D uint32_t block_exclusive_scan(uint32_t v, uint32_t* sum) {
    __shared__ uint32_t warp_tot[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint32_t t = lane < (int)(blockDim.x >> 5) ? warp_tot[lane] : 0u;
        uint32_t ti = t;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t u = __shfl_up_sync(0xffffffffu, ti, o);
            if (lane >= o) ti += u;
        }
        warp_tot[lane] = ti - t;  // exclusive warp offsets
        if (lane == 31) *sum = ti;
    }
    __syncthreads();
    uint32_t r = warp_tot[wid] + inc - v;
    __syncthreads();
    return r;
}

static __global__ void __launch_bounds__(kScanThreads)
k_scan_tiles(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint32_t n,
             uint32_t* __restrict__ tile_sums) {
    __shared__ uint32_t total;
    size_t base = (size_t)blockIdx.x * kScanTile + (size_t)threadIdx.x * kScanItems;
    uint32_t v[kScanItems], s = 0;
#pragma unroll
    for (int k = 0; k < kScanItems; k++) {
        v[k] = base + k < n ? in[base + k] : 0u;
        s += v[k];
    }
    uint32_t ex = block_exclusive_scan(s, &total);
#pragma unroll
    for (int k = 0; k < kScanItems; k++) {
        if (base + k < n) out[base + k] = ex;
        ex += v[k];
    }
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

// single block: exclusive scan of the tile sums in place; writes the grand total to *grand
static __global__ void __launch_bounds__(kScanThreads)
k_scan_sums(uint32_t* __restrict__ tile_sums, uint32_t ntiles, uint32_t* __restrict__ grand) {
    __shared__ uint32_t total;
    uint32_t carry = 0;
    for (uint32_t base = 0; base < ntiles; base += kScanThreads) {
        uint32_t i = base + threadIdx.x;
        uint32_t v = i < ntiles ? tile_sums[i] : 0u;
        uint32_t ex = block_exclusive_scan(v, &total);
        if (i < ntiles) tile_sums[i] = carry + ex;
        carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) *grand = carry;
}

// out[i] += tile offset; also mirrors the result into `copy` (the scatter cursors)
static __global__ void __launch_bounds__(kScanThreads)
k_scan_add(uint32_t* __restrict__ out, uint32_t* __restrict__ copy, uint32_t n,
           const uint32_t* __restrict__ tile_sums) {
    size_t base = (size_t)blockIdx.x * kScanTile + (size_t)threadIdx.x * kScanItems;
    uint32_t off = tile_sums[blockIdx.x];
#pragma unroll
    for (int k = 0; k < kScanItems; k++)
        if (base + k < n) {
            uint32_t v = out[base + k] + off;
            out[base + k] = v;
            copy[base + k] = v;
        }
}

// ---------------------------------------------------------------------------- shared-memory radix partition
// Large single MSMs sort their (bucket, point) pairs in two most-significant-digit passes instead of one
// returning global atomic per pair (k_digits<SCATTER>, bound by L2 atomic round trips: ncu long-scoreboard).
// The exact bucket offsets are already known from the histogram + scan, so every coarse bin (2^lb
// consecutive buckets) owns a contiguous range of the output and no pass needs its own global histogram.
//
//   pass 1  k_partition_coarse: a block takes a tile of kPartTile scalars, reduces them once into shared
//           memory (SoA words + the per-window carry bits of the signed recoding), then for each window:
//           shared-memory histogram over the window's coarse bins (atomicAdd returns the rank inside the
//           block), block scan, ONE global atomic per (block, bin) to reserve a run in the bin's range, the
//           pairs are grouped by bin in shared memory and written out as coalesced runs into `part`.
//   pass 2  k_partition_fine: a block takes kFineTile consecutive pairs of `part` (one or two coarse bins),
//           ranks them per bucket in a shared-memory histogram, reserves a run per (block, bucket) with one
//           global atomic on the bucket cursor, groups the pairs by bucket in shared memory and writes them
//           to their final place in `sorted` as coalesced runs.  Pairs whose bucket lies beyond the shared
//           histogram (sparse inputs) take one global atomic each.
#ifndef PORLA_PART_THREADS
#define PORLA_PART_THREADS 512
#endif
#ifndef PORLA_PART_PER_THREAD
#define PORLA_PART_PER_THREAD 4
#endif
#ifndef PORLA_PART_MIN_BLOCKS
#define PORLA_PART_MIN_BLOCKS 2
#endif
constexpr int kPartThreads = PORLA_PART_THREADS;
constexpr int kPartPerThread = PORLA_PART_PER_THREAD;
constexpr int kPartTile = kPartThreads * kPartPerThread;   // 2048 scalars: 64 KB of reduced words in smem
constexpr int kPartMaxBins = 1024;                         // coarse bins per window
constexpr int kFineThreads = 512;
constexpr int kFinePerThread = 8;
constexpr int kFineTile = kFineThreads * kFinePerThread;   // 4096 pairs
constexpr uint32_t kFineHist = 4096;                       // shared histogram entries of pass 2
constexpr uint32_t kMetaSkip = 1u << 30, kMetaFlip = 1u << 31, kMetaFlip2 = 1u << 29;
constexpr uint32_t kBigBin = 34816;   // pairs per bin k_fine_smem keeps in shared memory (6 B each: 204 KB + the histogram)

static __global__ void k_init_coarse(const uint32_t* __restrict__ offsets, uint32_t nbt, int lb, uint32_t ncoarse,
                                     uint32_t* __restrict__ coarse_cursor) {
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < ncoarse) coarse_cursor[g] = offsets[(size_t)g << lb];
}

constexpr int kPartCoarseSmem = (9 * kPartTile + 2 * kPartMaxBins) * 4 + kPartTile * 8;   // dynamic shared memory: the layout below
template <class C, bool GLV>
__global__ void __launch_bounds__(kPartThreads, PORLA_PART_MIN_BLOCKS)
k_partition_coarse(const uint8_t* __restrict__ scalars, int big_endian, const uint8_t* __restrict__ inf_flags,
                   MsmShape sh, int lb, uint32_t* __restrict__ coarse_cursor, uint2* __restrict__ part) {
    extern __shared__ uint32_t smem[];
    uint32_t* sw = smem;                                   // [8][kPartTile] reduced scalar words
    uint32_t* meta = sw + 8 * kPartTile;                   // carry bit per window | skip | flip
    uint32_t* cnt = meta + kPartTile;                      // [kPartMaxBins] counts, then local offsets
    uint32_t* delta = cnt + kPartMaxBins;                  // [kPartMaxBins] reserved global base - local offset
    uint2* stage = reinterpret_cast<uint2*>(delta + kPartMaxBins);   // [kPartTile] pairs grouped by bin
    __shared__ uint32_t s_total;
    const uint32_t ncw = sh.nbuckets >> lb;                // coarse bins per window (<= kPartMaxBins)
    const uint32_t half = 1u << (sh.c - 1);
    const uint32_t mask = (1u << sh.c) - 1u;
    const uint32_t tile0 = blockIdx.x * kPartTile;
    // ---- reduce the tile's scalars once, note the carries of the signed recoding
#pragma unroll 1
    for (int q = 0; q < kPartPerThread; q++) {
        const uint32_t p = q * kPartThreads + threadIdx.x;
        const uint32_t i = tile0 + p;
        uint32_t m = kMetaSkip;
        uint32_t s[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};     // GLV: |k1| in s[0..3], |k2| in s[4..7]
        if (i < sh.n && !(inf_flags && inf_flags[i])) {
            if constexpr (GLV) {
                uint32_t n1, n2;
                glv_scalar<C>(scalars, i, big_endian, s, s + 4, n1, n2);
                m = (n1 ? kMetaFlip : 0u) | (n2 ? kMetaFlip2 : 0u);
            } else {
                m = canonical_scalar<C>(scalars, i, big_endian, s) ? kMetaFlip : 0u;
            }
        }
#pragma unroll
        for (int k = 0; k < 8; k++) sw[k * kPartTile + p] = s[k];
        meta[p] = m;
    }
    // ---- one window at a time
    const uint32_t ept = (ncw + kPartThreads - 1) / kPartThreads;   // bins per thread in the scan (<= 2)
    // The windows are visited in order and a thread meets the same kPartPerThread scalars in every window, so the carries of
    // the signed recoding live in registers across the loop (round 1 precomputed them per scalar with a dynamically indexed
    // limb array: ~600 instructions per scalar of compare / select chains, a quarter of this kernel).
    uint32_t carry[kPartPerThread];
#pragma unroll
    for (int q = 0; q < kPartPerThread; q++) carry[q] = 0;
    for (int w = 0; w < sh.nwin; w++) {
        for (uint32_t b = threadIdx.x; b < ncw; b += kPartThreads) cnt[b] = 0;
        __syncthreads();
        const int h = GLV && w >= sh.glv_wh ? 1 : 0;          // GLV: second half, phi(P_i), the first half's buckets
        const int wl = w - h * (GLV ? sh.glv_wh : 0);
        const uint32_t pos = (uint32_t)wl * sh.c;
        const uint32_t word = (pos >> 5) + (GLV ? 4u * h : 0u), sft = pos & 31;
        const uint32_t word_end = GLV ? 4u * h + 4u : 8u;       // first limb past the value being recoded
        const uint32_t key0 = sh.fixed_n ? 0u : (uint32_t)wl * sh.nbuckets;
        const uint32_t flip_bit = h ? 29u : 31u;
        if (GLV && wl == 0) {
#pragma unroll
            for (int q = 0; q < kPartPerThread; q++) carry[q] = 0;     // second half: a new value
        }
        // packed per item: bucket (20 bits) | rank within (block, bin) (11 bits) | sign
        uint32_t item[kPartPerThread];
#pragma unroll
        for (int q = 0; q < kPartPerThread; q++) {
            const uint32_t p = q * kPartThreads + threadIdx.x;
            const uint32_t m = meta[p];
            item[q] = 0xffffffffu;
            if (!(m & kMetaSkip)) {
                uint32_t lo = word < word_end ? sw[word * kPartTile + p] : 0u;
                uint32_t hi = word + 1 < word_end ? sw[(word + 1) * kPartTile + p] : 0u;
                uint32_t d = (__funnelshift_r(lo, hi, sft) & mask) + carry[q];
                uint32_t dneg = d > half;
                carry[q] = dneg;
                uint32_t mag = dneg ? ((1u << sh.c) - d) : d;
                if (mag != 0) {
                    uint32_t r = atomicAdd(&cnt[(mag - 1) >> lb], 1u);     // r < kPartTile = 2^11
                    item[q] = (mag - 1) | (r << 20) | ((dneg ^ ((m >> flip_bit) & 1u)) << 31);
                }
            }
        }
        __syncthreads();
        // exclusive scan of the bin counts (local offsets), one global reservation per non-empty bin
        {
            uint32_t v[(kPartMaxBins + kPartThreads - 1) / kPartThreads], sum = 0;
            const uint32_t b0 = threadIdx.x * ept;
            for (uint32_t k = 0; k < ept; k++) {
                v[k] = b0 + k < ncw ? cnt[b0 + k] : 0u;
                sum += v[k];
            }
            uint32_t ex = block_exclusive_scan(sum, &s_total);
            for (uint32_t k = 0; k < ept; k++) {
                if (b0 + k < ncw) {
                    cnt[b0 + k] = ex;
                    delta[b0 + k] = v[k] ? atomicAdd(&coarse_cursor[(key0 >> lb) + b0 + k], v[k]) - ex : 0u;
                }
                ex += v[k];
            }
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < kPartPerThread; q++) {
            if (item[q] == 0xffffffffu) continue;
            const uint32_t bucket = item[q] & 0xfffffu, r = (item[q] >> 20) & 0x7ffu, neg = item[q] >> 31;
            const uint32_t pidx = tile0 + q * kPartThreads + threadIdx.x + (h ? sh.phi_off : 0u);
            stage[cnt[bucket >> lb] + r] =
                make_uint2(key0 + bucket, (sh.fixed_n ? (uint32_t)w * sh.fixed_n + pidx : pidx) | (neg << 31));
        }
        __syncthreads();
        const uint32_t total = s_total;
        for (uint32_t j = threadIdx.x; j < total; j += kPartThreads) {
            const uint2 e = stage[j];
            part[delta[(e.x - key0) >> lb] + j] = e;
        }
    }
}

PORLA_D bool bin_is_big(const uint32_t* __restrict__ coarse_off, uint32_t bin) {
    return coarse_off[bin + 1] - coarse_off[bin] > kBigBin;
}

constexpr int kPartFineSmem = 2 * kFineHist * 4 + kFineTile * 8;   // dynamic shared memory: the layout below
// kBigOnly: only the pairs of bins above kBigBin pairs, for the sort without the exact histogram (cursor = the offsets
// k_big_scan wrote; tiles without such pairs return at once).  Otherwise coarse_off is not read.
template <bool kBigOnly>
static __global__ void __launch_bounds__(kFineThreads, 3)
k_partition_fine(const uint2* __restrict__ part, const uint32_t* __restrict__ total_pairs, const uint32_t* __restrict__ coarse_off,
                 int lb, uint32_t* __restrict__ cursor, uint2* __restrict__ sorted) {
    extern __shared__ uint32_t smem[];
    uint32_t* cnt = smem;                                   // [kFineHist] counts, then local offsets
    uint32_t* delta = cnt + kFineHist;                      // [kFineHist] reserved global base - local offset
    uint2* stage = reinterpret_cast<uint2*>(delta + kFineHist);   // [kFineTile] pairs grouped by bucket
    __shared__ uint32_t s_total;
    const uint32_t M = *total_pairs;
    const uint64_t lo64 = (uint64_t)blockIdx.x * kFineTile;
    if (lo64 >= M) return;
    const uint32_t lo = (uint32_t)lo64;
    const uint32_t hi = M - lo > (uint32_t)kFineTile ? lo + kFineTile : M;
    const uint32_t bin_lo = __ldg(&part[lo].x) >> lb;
    if constexpr (kBigOnly) {   // the tile covers the bins of its first .. last pair
        const uint32_t bin_hi = __ldg(&part[hi - 1].x) >> lb;
        bool any = false;
        for (uint32_t b = bin_lo; b <= bin_hi && !any; b++) any = bin_is_big(coarse_off, b);
        if (!any) return;
    }
    for (uint32_t b = threadIdx.x; b < kFineHist; b += kFineThreads) cnt[b] = 0;
    const uint32_t kbase = bin_lo << lb;
    __syncthreads();
    uint2 e[kFinePerThread];
    uint32_t rank[kFinePerThread];
#pragma unroll
    for (int q = 0; q < kFinePerThread; q++) {
        const uint32_t idx = lo + q * kFineThreads + threadIdx.x;
        e[q] = make_uint2(0xffffffffu, 0u);
        if (idx < hi) {
            const uint2 v = __ldg(&part[idx]);
            if (!kBigOnly || bin_is_big(coarse_off, v.x >> lb)) {
                e[q] = v;
                const uint32_t rel = v.x - kbase;      // pass 1 keeps coarse bins in order, so rel >= 0
                if (rel < kFineHist) rank[q] = atomicAdd(&cnt[rel], 1u);
            }
        }
    }
    __syncthreads();
    {
        constexpr uint32_t ept = kFineHist / kFineThreads;   // 8
        uint32_t v[ept], sum = 0;
        const uint32_t b0 = threadIdx.x * ept;
#pragma unroll
        for (uint32_t k = 0; k < ept; k++) {
            v[k] = cnt[b0 + k];
            sum += v[k];
        }
        uint32_t ex = block_exclusive_scan(sum, &s_total);
#pragma unroll
        for (uint32_t k = 0; k < ept; k++) {
            cnt[b0 + k] = ex;
            delta[b0 + k] = v[k] ? atomicAdd(&cursor[kbase + b0 + k], v[k]) - ex : 0u;
            ex += v[k];
        }
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < kFinePerThread; q++) {
        if (e[q].x == 0xffffffffu) continue;
        const uint32_t rel = e[q].x - kbase;
        if (rel < kFineHist) stage[cnt[rel] + rank[q]] = e[q];
        else sorted[atomicAdd(&cursor[e[q].x], 1u)] = e[q];
    }
    __syncthreads();
    const uint32_t total = s_total;
    for (uint32_t j = threadIdx.x; j < total; j += kFineThreads) {
        const uint2 x = stage[j];
        sorted[delta[x.x - kbase] + j] = x;
    }
}

// ---------------------------------------------------------------------------- sort without the exact histogram (round 2: the
// default radix path when the coarse bins fit a block, see msm_impl.cuh and profiles/r02b_sort_without_exact_histogram.txt)
// The exact bucket histogram (k_digits<COUNT>: one global atomic per pair, 218 M of them at 2^24) exists only to give every
// bucket its output range.  The radix path does not need it: a COARSE histogram (one counter per 2^lb consecutive buckets,
// kept in shared memory while a block walks its share of the scalars) is enough to place the coarse bins, and each coarse
// bin is then sorted by ONE block that counts, scans and scatters its own 2^lb buckets in shared memory.
//   k_coarse_count   recode every scalar, shared-memory histogram over (window, coarse bin), a few global atomics per block
//   k_coarse_scan    exclusive scan of the <= 28 k coarse counters -> bin offsets, partition cursors, total pair count
//   k_partition_coarse (above) writes the pairs grouped by coarse bin into `part`
//   k_fine_smem      block b owns coarse bin b: histogram of its buckets, scan, placement in shared memory, ordered write-out
// Skewed inputs (a constant scalar, 31-bit scalars' empty top windows ...) put up to all pairs of a window into one coarse
// bin; bins above kBigBin pairs are left to the tile-based route, which is the round-1 fine pass preceded by its own
// counting pass over the same tiles (k_big_count, k_big_scan, k_partition_fine<true>) and costs nothing when no bin is big.
constexpr int kCoarseCountThreads = 512;
constexpr int kFineLocalThreads = 256;
constexpr uint32_t kFineLocalBuckets = 1024;   // 2^lb <= 2^10 buckets per coarse bin (c <= 20)

constexpr int kCoarseCountSmem = 160 << 10;   // dynamic shared memory limit: one counter per coarse bin of every window
template <class C, bool GLV>
__global__ void __launch_bounds__(kCoarseCountThreads)
k_coarse_count(const uint8_t* __restrict__ scalars, int big_endian, const uint8_t* __restrict__ inf_flags, MsmShape sh, int lb,
               uint32_t ncoarse, uint32_t* __restrict__ coarse_count) {
    extern __shared__ uint32_t smem[];   // [ncoarse]
    for (uint32_t b = threadIdx.x; b < ncoarse; b += blockDim.x) smem[b] = 0;
    __syncthreads();
    const uint32_t half = 1u << (sh.c - 1);
    const uint32_t mask = (1u << sh.c) - 1u;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < sh.n; i += (uint64_t)gridDim.x * blockDim.x) {
        if (inf_flags && inf_flags[i]) continue;
        uint32_t s[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};     // GLV: |k1| in s[0..3], |k2| in s[4..7]
        if constexpr (GLV) {
            uint32_t n1, n2;
            glv_scalar<C>(scalars, i, big_endian, s, s + 4, n1, n2);
        } else {
            canonical_scalar<C>(scalars, i, big_endian, s);
        }
        // Walk the value word by word with a 64-bit shift register: the limbs are indexed statically (a dynamically indexed
        // register array cost ~40 instructions of compare / select chains per window here), one c-bit digit per turn.
        const int halves = GLV ? 2 : 1, words = GLV ? 4 : 8, wins = GLV ? sh.glv_wh : sh.nwin;
#pragma unroll
        for (int h = 0; h < halves; h++) {
            uint64_t acc = 0;
            int have = 0, wl = 0;
            uint32_t carry = 0;
#pragma unroll
            for (int k = 0; k <= words; k++) {
                const uint32_t limb = k < words ? s[h * 4 + k] : 0u;      // one zero word past the top: the last digits
                acc |= (uint64_t)limb << have;
                have += 32;
                while (wl < wins && (have >= sh.c || k == words)) {
                    const uint32_t d = ((uint32_t)acc & mask) + carry;
                    acc >>= sh.c;
                    have -= sh.c;
                    const uint32_t dneg = d > half;
                    carry = dneg;
                    const uint32_t mag = dneg ? ((1u << sh.c) - d) : d;
                    if (mag != 0) {
                        const uint32_t key0 = sh.fixed_n ? 0u : (uint32_t)wl * sh.nbuckets;
                        atomicAdd(&smem[(key0 + (mag - 1)) >> lb], 1u);
                    }
                    wl++;
                }
            }
        }
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < ncoarse; b += blockDim.x)
        if (smem[b]) atomicAdd(&coarse_count[b], smem[b]);
}

// single block: coarse_off[0..ncoarse] = exclusive scan of coarse_count, cursor copy, total
static __global__ void __launch_bounds__(1024)
k_coarse_scan(const uint32_t* __restrict__ coarse_count, uint32_t ncoarse, uint32_t* __restrict__ coarse_off,
              uint32_t* __restrict__ coarse_cursor, uint32_t* __restrict__ grand) {
    __shared__ uint32_t total;
    uint32_t carry = 0;
    for (uint32_t base = 0; base < ncoarse; base += blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = i < ncoarse ? coarse_count[i] : 0u;
        const uint32_t ex = block_exclusive_scan(v, &total);
        if (i < ncoarse) {
            coarse_off[i] = carry + ex;
            coarse_cursor[i] = carry + ex;
        }
        carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        coarse_off[ncoarse] = carry;
        *grand = carry;
    }
}

// Block b sorts coarse bin b (pairs part[off[b] .. off[b+1])) by bucket into the same range of `sorted`, THROUGH SHARED MEMORY:
// the bin is read once for its bucket histogram and once more (from L2: one block per SM keeps 148 bins = 38 MB in flight) to
// place every pair's 32-bit point word and 16-bit local bucket at its final position in shared memory, then written out in
// order -- whole lines, no global atomics, no scattered 8-byte stores (the first version of this kernel scattered straight to
// global memory: 3.85 ms at 2^24 with 2.6 % of the issue slots used, 5.1 GB read and 3.5 GB written for 1.75 GB of pairs;
// profiles/r02b_sort_without_exact_histogram.txt).  Six bytes of shared memory per pair: bins of up to kBigBin pairs.
constexpr int kFineSmemThreads = 1024;
constexpr int kFineLocalSmem = kBigBin * 6 + kFineLocalBuckets * 4;   // dynamic shared memory: the layout below
static __global__ void __launch_bounds__(kFineSmemThreads, 1)
k_fine_smem(const uint2* __restrict__ part, const uint32_t* __restrict__ coarse_off, int lb, uint2* __restrict__ sorted,
            uint4* __restrict__ zero_buckets) {
    extern __shared__ uint32_t smem[];
    uint32_t* out_y = smem;                                              // [kBigBin] point word of the pair at each position
    uint16_t* out_b = reinterpret_cast<uint16_t*>(out_y + kBigBin);      // [kBigBin] its bucket within the bin
    uint32_t* hist = reinterpret_cast<uint32_t*>(out_b + kBigBin);       // [kFineLocalBuckets] counts, then cursors
    __shared__ uint32_t total;
    const uint32_t start = coarse_off[blockIdx.x], cnt = coarse_off[blockIdx.x + 1] - start;
    // zero_buckets != nullptr: this pass also writes the EMPTY buckets of its bin (128-byte records of zeros = infinity), which
    // replaces the memset of the whole bucket array (872 MB at 2^24) by the few buckets that really are empty
    uint4* zb = zero_buckets ? zero_buckets + ((size_t)blockIdx.x << lb) * 8 : nullptr;
    if (cnt == 0) {
        if (zb)
            for (uint32_t j = threadIdx.x; j < (8u << lb); j += kFineSmemThreads) zb[j] = make_uint4(0u, 0u, 0u, 0u);
        return;
    }
    if (cnt > kBigBin) return;                              // k_big_scan zeroes this bin's empty buckets
    const uint32_t bmask = (1u << lb) - 1u;
    const uint2* src = part + start;
    for (uint32_t b = threadIdx.x; b < kFineLocalBuckets; b += kFineSmemThreads) hist[b] = 0;
    __syncthreads();
    // 1. histogram (four loads in flight per thread)
    for (uint32_t j0 = 0; j0 < cnt; j0 += 4 * kFineSmemThreads) {
        uint32_t key[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t j = j0 + k * kFineSmemThreads + threadIdx.x;
            key[k] = j < cnt ? __ldg(&src[j].x) : 0xffffffffu;
        }
#pragma unroll
        for (int k = 0; k < 4; k++)
            if (j0 + k * kFineSmemThreads + threadIdx.x < cnt) atomicAdd(&hist[key[k] & bmask], 1u);
    }
    __syncthreads();
    // 2. exclusive scan of the (at most 1024) bucket counts: cursors
    {
        const uint32_t v = threadIdx.x < kFineLocalBuckets ? hist[threadIdx.x] : 0u;
        if (zb && v == 0 && threadIdx.x <= bmask) {
#pragma unroll
            for (int k = 0; k < 8; k++) zb[(size_t)threadIdx.x * 8 + k] = make_uint4(0u, 0u, 0u, 0u);
        }
        const uint32_t ex = block_exclusive_scan(v, &total);
        if (threadIdx.x < kFineLocalBuckets) hist[threadIdx.x] = ex;
    }
    __syncthreads();
    // 3. place
    for (uint32_t j0 = 0; j0 < cnt; j0 += 4 * kFineSmemThreads) {
        uint2 e[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t j = j0 + k * kFineSmemThreads + threadIdx.x;
            e[k] = j < cnt ? __ldg(&src[j]) : make_uint2(0u, 0u);
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (j0 + k * kFineSmemThreads + threadIdx.x < cnt) {
                const uint32_t b = e[k].x & bmask;
                const uint32_t pos = atomicAdd(&hist[b], 1u);
                out_y[pos] = e[k].y;
                out_b[pos] = (uint16_t)b;
            }
        }
    }
    __syncthreads();
    // 4. write out in order; all pairs of the bin share the bucket id above the low lb bits
    const uint32_t key_hi = __ldg(&src[0].x) & ~bmask;
    uint2* dst = sorted + start;
    for (uint32_t j = threadIdx.x; j < cnt; j += kFineSmemThreads) dst[j] = make_uint2(key_hi | out_b[j], out_y[j]);
}

// ---- bins above kBigBin pairs: the tile-based fine pass with its own counting pass
static __global__ void __launch_bounds__(kFineThreads)
k_big_count(const uint2* __restrict__ part, const uint32_t* __restrict__ total_pairs, const uint32_t* __restrict__ coarse_off,
            int lb, uint32_t* __restrict__ counters) {
    const uint32_t M = *total_pairs;
    const uint64_t lo64 = (uint64_t)blockIdx.x * kFineTile;
    if (lo64 >= M) return;
    const uint32_t lo = (uint32_t)lo64;
    const uint32_t hi = M - lo > (uint32_t)kFineTile ? lo + kFineTile : M;
    // the tile covers the bins of its first .. last pair (pass 1 keeps the coarse bins in order)
    const uint32_t bin_lo = __ldg(&part[lo].x) >> lb, bin_hi = __ldg(&part[hi - 1].x) >> lb;
    bool any = false;
    for (uint32_t b = bin_lo; b <= bin_hi && !any; b++) any = bin_is_big(coarse_off, b);
    if (!any) return;
    // shared-memory histogram of the tile (a constant scalar sends every pair of the tile to ONE bucket), one global atomic
    // per (tile, bucket)
    __shared__ uint32_t hist[kFineHist];
    for (uint32_t b = threadIdx.x; b < kFineHist; b += kFineThreads) hist[b] = 0;
    const uint32_t kbase = bin_lo << lb;
    __syncthreads();
    for (uint32_t idx = lo + threadIdx.x; idx < hi; idx += kFineThreads) {
        const uint32_t key = __ldg(&part[idx].x);
        if (!bin_is_big(coarse_off, key >> lb)) continue;
        const uint32_t rel = key - kbase;
        if (rel < kFineHist) atomicAdd(&hist[rel], 1u);
        else atomicAdd(&counters[key], 1u);
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < kFineHist; b += kFineThreads)
        if (hist[b]) atomicAdd(&counters[kbase + b], hist[b]);
}

// block b: if bin b is big, counters[b << lb ..] <- its output offsets (bin start + exclusive prefix of the counts)
static __global__ void __launch_bounds__(kFineLocalThreads)
k_big_scan(const uint32_t* __restrict__ coarse_off, int lb, uint32_t* __restrict__ counters, uint4* __restrict__ zero_buckets) {
    __shared__ uint32_t total;
    if (!bin_is_big(coarse_off, blockIdx.x)) return;
    const uint32_t nb = 1u << lb;
    uint32_t* c = counters + ((size_t)blockIdx.x << lb);
    uint4* zb = zero_buckets ? zero_buckets + ((size_t)blockIdx.x << lb) * 8 : nullptr;     // see k_fine_smem
    uint32_t carry = coarse_off[blockIdx.x];
    for (uint32_t base = 0; base < nb; base += kFineLocalThreads) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = i < nb ? c[i] : 0u;
        if (zb && i < nb && v == 0) {
#pragma unroll
            for (int k = 0; k < 8; k++) zb[(size_t)i * 8 + k] = make_uint4(0u, 0u, 0u, 0u);
        }
        const uint32_t ex = block_exclusive_scan(v, &total);
        if (i < nb) c[i] = carry + ex;
        carry += total;
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------- accumulation
// Load-balanced segmented accumulation.  `sorted` holds the M (bucket id, point index | sign << 31)
// pairs grouped by bucket.  Thread t owns the fixed-length slice [t*L, (t+1)*L) regardless of where
// bucket boundaries fall, so every thread performs the same number of mixed additions whatever
// the digit distribution (31-bit audit coefficients, the short top window, repeated scalars).
// A bucket that lies wholly inside one slice is written straight to buckets[]; a bucket cut by a
// slice boundary leaves a partial sum: part_head[t] (the bucket continues from slice t-1) or
// part_tail[t] (it continues into slice t+1).  k_stitch then adds the partials of each cut bucket.
constexpr int kAccThreads = 128;
#ifndef PORLA_ACC_MIN_BLOCKS
#define PORLA_ACC_MIN_BLOCKS 4
#endif

// e = point index | sign << 31.  Indices from phi_off on (phi_off != 0) address the endomorphism image of entry
// index - phi_off: x from the beta*x array, y from the table record.
template <class C>
PORLA_D Affine<typename C::F> load_signed_point(const Affine<typename C::F>* __restrict__ points,
                                                const typename C::F* __restrict__ phi_x, uint32_t phi_off, uint32_t e) {
    using F = typename C::F;
    const uint32_t idx = e & 0x7fffffffu;
    const bool image = C::kGlv && phi_off != 0 && idx >= phi_off;
    const uint32_t j = image ? idx - phi_off : idx;
    const uint4* sx = image ? reinterpret_cast<const uint4*>(phi_x + j) : reinterpret_cast<const uint4*>(points + j);
    const uint4* sy = reinterpret_cast<const uint4*>(points + j) + 2;
    Affine<F> p;
    uint4* d = reinterpret_cast<uint4*>(&p);
    d[0] = __ldg(sx);
    d[1] = __ldg(sx + 1);
    d[2] = __ldg(sy);
    d[3] = __ldg(sy + 1);
    if (e >> 31) p.y = p.y.neg();
    return p;
}

// `into` != 0 (a later part of a streamed MSM, msm_host_pipelined): the buckets already hold the sums of the earlier parts;
// the thread that owns the START of a bucket's run continues from that value (one more mixed addition per bucket and part)
// instead of starting from the first point, so that all parts of the MSM share one bucket set and one reduction.  The
// stored value only seeds the accumulator: the loop keeps ONE call site of the mixed addition (three inlined copies of it
// overflow the instruction cache -- measured: 2.4x slower per pair).
template <class F>
PORLA_D XYZZ<F> bucket_seed(const XYZZ<F>* __restrict__ buckets, uint32_t key, int into) {
    XYZZ<F> acc = XYZZ<F>::inf();
    if (into) {   // plain loads: written by the previous part's kernels on this stream
        const uint4* s = reinterpret_cast<const uint4*>(buckets + key);
        uint4* d = reinterpret_cast<uint4*>(&acc);
#pragma unroll
        for (int i = 0; i < 8; i++) d[i] = s[i];
    }
    return acc;
}

template <class C>
__global__ void __launch_bounds__(kAccThreads, PORLA_ACC_MIN_BLOCKS)
k_accumulate(const Affine<typename C::F>* __restrict__ points, const typename C::F* __restrict__ phi_x, uint32_t phi_off,
             const uint2* __restrict__ sorted, const uint32_t* __restrict__ total_pairs, uint32_t L,
             XYZZ<typename C::F>* __restrict__ buckets, XYZZ<typename C::F>* __restrict__ part_head,
             XYZZ<typename C::F>* __restrict__ part_tail, int into) {
    using F = typename C::F;
    const uint32_t M = *total_pairs;
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t start64 = (uint64_t)t * L;
    if (start64 >= M) return;
    const uint32_t start = (uint32_t)start64;
    const uint32_t end = (M - start > L) ? start + L : M;
    const uint32_t prev_key = start > 0 ? __ldg(&sorted[start - 1].x) : 0xffffffffu;
    const uint32_t next_key = end < M ? __ldg(&sorted[end].x) : 0xffffffffu;

    uint32_t key = __ldg(&sorted[start].x);
    bool first = true;  // still inside the first bucket of this slice
    // the run's first pair lies in this slice unless the bucket continues from the left (then the owner slice seeded it)
    XYZZ<F> acc = prev_key == key ? XYZZ<F>::inf() : bucket_seed<F>(buckets, key, into);
    for (uint32_t pos = start; pos < end; ++pos) {
        const uint2 e = __ldg(&sorted[pos]);
        const Affine<F> q = load_signed_point<C>(points, phi_x, phi_off, e.y);
        if (e.x != key) {
            if (first && prev_key == key) st16(part_head + t, acc);
            else st16(buckets + key, acc);
            first = false;
            key = e.x;
            acc = bucket_seed<F>(buckets, key, into);
        }
        if (acc.is_inf()) acc = XYZZ<F>{q.x, q.y, F::one(), F::one()};
        else acc.madd_finite(q);
    }
    if (first && prev_key == key) st16(part_head + t, acc);        // continues from the left (maybe also to the right)
    else if (next_key == key) st16(part_tail + t, acc);            // starts here, continues to the right
    else st16(buckets + key, acc);
}

// One thread per slice boundary owner: slice t owns the cut bucket that STARTS inside it and runs on
// into slice t+1; it adds part_tail[t] and the part_head[] of every following slice the bucket
// covers.  Buckets longer than L * kStitchSerial pairs are finished by k_stitch_long (a block each).
constexpr uint32_t kStitchSerial = 48;       // throughput setting: many cut buckets, every thread busy
constexpr uint32_t kStitchSerialSmall = 8;   // latency setting: few slices in total, hand long runs to a block early

template <class C>
__global__ void __launch_bounds__(64)
k_stitch(const uint2* __restrict__ sorted, const uint32_t* __restrict__ total_pairs, uint32_t L,
         XYZZ<typename C::F>* __restrict__ buckets, const XYZZ<typename C::F>* __restrict__ part_head,
         const XYZZ<typename C::F>* __restrict__ part_tail, uint32_t* __restrict__ long_count,
         uint2* __restrict__ long_runs, uint32_t serial_limit) {
    using F = typename C::F;
    const uint32_t M = *total_pairs;
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t start64 = (uint64_t)t * L;
    if (start64 >= M) return;
    const uint32_t start = (uint32_t)start64;
    if (M - start <= L) return;                       // last slice: nothing to its right
    const uint32_t end = start + L;
    const uint32_t key = __ldg(&sorted[end - 1].x);
    if (__ldg(&sorted[end].x) != key) return;         // no bucket is cut at this boundary
    if (__ldg(&sorted[start].x) == key && start > 0 && __ldg(&sorted[start - 1].x) == key) return;  // not the owner
    // how many following slices does the bucket touch?  (binary search would also do; runs are short)
    const uint32_t nslices = (uint32_t)(((uint64_t)M + L - 1) / L);
    uint32_t u = t + 1, cnt = 0;
    XYZZ<F> acc = ld16(part_tail + t);
    for (;;) {
        if (cnt == serial_limit) {                    // hand the rest to the cooperative kernel
            st16(buckets + key, acc);
            uint32_t slot = atomicAdd(long_count, 1u);
            long_runs[slot] = make_uint2(key, u);
            return;
        }
        acc.add(ld16(part_head + u));
        cnt++;
        // does slice u lie wholly inside the bucket and continue?
        uint32_t uend = (u + 1 < nslices) ? (u + 1) * L : M;
        if (u + 1 < nslices && __ldg(&sorted[uend - 1].x) == key && __ldg(&sorted[uend].x) == key) u++;
        else break;
    }
    st16(buckets + key, acc);
}

// Cooperative tail for very long buckets (skewed inputs such as a constant scalar): block b takes
// long_runs[b] = (bucket, first unprocessed slice u0); its threads add part_head[u0 + j], j strided,
// then a shared-memory tree; the result is added to what k_stitch already stored.
constexpr int kLongThreads = 128;

template <class C>
__global__ void __launch_bounds__(kLongThreads)
k_stitch_long(const uint2* __restrict__ sorted, const uint32_t* __restrict__ total_pairs, uint32_t L,
              XYZZ<typename C::FC>* __restrict__ buckets, const XYZZ<typename C::FC>* __restrict__ part_head,
              const uint32_t* __restrict__ long_count, const uint2* __restrict__ long_runs) {
    using F = typename C::FC;
    __shared__ XYZZ<F> sh[kLongThreads];
    __shared__ uint32_t s_last;
    const uint32_t M = *total_pairs;
    const uint32_t nruns = *long_count;
    const uint32_t nslices = (uint32_t)(((uint64_t)M + L - 1) / L);
    for (uint32_t r = blockIdx.x; r < nruns; r += gridDim.x) {
        const uint32_t key = long_runs[r].x, u0 = long_runs[r].y;
        if (threadIdx.x == 0) {
            // last slice touched by the bucket: binary search for the last pair with this key
            uint32_t lo = u0 * L, hi = M;  // sorted[lo].x == key (slice u0 starts inside the bucket)
            while (hi - lo > 1) {
                uint32_t mid = lo + (hi - lo) / 2;
                if (__ldg(&sorted[mid].x) == key) lo = mid;
                else hi = mid;
            }
            s_last = lo / L;
        }
        __syncthreads();
        const uint32_t last = s_last < nslices ? s_last : nslices - 1;
        XYZZ<F> acc = XYZZ<F>::inf();
        for (uint32_t u = u0 + threadIdx.x; u <= last; u += kLongThreads) acc.add(ld16(part_head + u));
        sh[threadIdx.x] = acc;
        __syncthreads();
        for (int o = kLongThreads / 2; o > 0; o >>= 1) {
            if ((int)threadIdx.x < o) {
                XYZZ<F> a = sh[threadIdx.x];
                a.add(sh[threadIdx.x + o]);
                sh[threadIdx.x] = a;
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            XYZZ<F> a = ld16(buckets + key);
            a.add(sh[0]);
            st16(buckets + key, a);
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------- bucket reduction
// Window slot s owns buckets[s*nb .. (s+1)*nb); bucket k has weight k+1.  Thread t of the slot
// takes the chunk [t*chunk, (t+1)*chunk): running sums give sum_k (k-lo+1) B_k and S = sum_k B_k;
// adding lo*S (small double-and-add) yields the chunk's weighted sum.  A shared-memory tree then
// leaves one partial per block:  partials[s * blocks_per_slot + blockIdx.x].
constexpr int kRedThreads = 64;

template <class C>
__global__ void __launch_bounds__(kRedThreads)
k_reduce(const XYZZ<typename C::FC>* __restrict__ buckets, uint32_t nb, uint32_t chunk,
         uint32_t threads_per_slot, uint32_t total_slots, XYZZ<typename C::FC>* __restrict__ partials) {
    using F = typename C::FC;
    __shared__ XYZZ<F> sh[kRedThreads];
    // Geometry (1-D grid; gridDim.y would cap the number of window slots at 65535):
    //   threads_per_slot >= 64: blocks_per_slot blocks per slot, one partial per block;
    //   threads_per_slot  < 64 (a power of two; small windows of batched MSMs): 64/threads_per_slot
    //   slots per block, the shared-memory tree stops at the slot boundary, one partial per slot.
    uint32_t slot, t, group;
    size_t out_index;
    if (threads_per_slot >= kRedThreads) {
        const uint32_t blocks_per_slot = (threads_per_slot + kRedThreads - 1) / kRedThreads;
        slot = blockIdx.x / blocks_per_slot;
        const uint32_t blk = blockIdx.x - slot * blocks_per_slot;
        t = blk * kRedThreads + threadIdx.x;
        group = kRedThreads;
        out_index = (size_t)slot * blocks_per_slot + blk;
    } else {
        const uint32_t slots_per_block = kRedThreads / threads_per_slot;
        slot = blockIdx.x * slots_per_block + threadIdx.x / threads_per_slot;
        t = threadIdx.x % threads_per_slot;
        group = threads_per_slot;
        out_index = slot;
    }
    XYZZ<F> acc = XYZZ<F>::inf();
    if (slot < total_slots && t < threads_per_slot) {
        const XYZZ<F>* base = buckets + (size_t)slot * nb;
        uint32_t lo = t * chunk;
        uint32_t hi = lo + chunk < nb ? lo + chunk : nb;
        XYZZ<F> run = XYZZ<F>::inf();
        for (uint32_t k = hi; k-- > lo;) {
            XYZZ<F> bk = ld16(base + k);
            run.add(bk);
            acc.add(run);
        }
        if (lo != 0) {
            XYZZ<F> w = mul_small(run, lo);
            acc.add(w);
        }
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
    const uint32_t local = threadIdx.x % group;
    for (uint32_t o = group / 2; o > 0; o >>= 1) {
        if (local < o) {
            XYZZ<F> a = sh[threadIdx.x];
            a.add(sh[threadIdx.x + o]);
            sh[threadIdx.x] = a;
        }
        __syncthreads();
    }
    if (local == 0 && slot < total_slots) st16(partials + out_index, sh[threadIdx.x]);
}

// ---------------------------------------------------------------------------- bucket reduction, scan form on quads (round 2)
// Below ~half a million buckets k_reduce is bound by the DEPTH of its dependent additions (6.9 us each on a lone warp), not
// by the multiplier pipe.  This form shortens every addition instead: four lanes per point (quad.cuh, 2.35 us per addition),
// and replaces the per-thread double-and-add weighting by scans:  sum_k (k + 1) B_k = sum_k R_k  with R_k = sum_{j >= k} B_j.
// A block of kQuadsPerBlock quads owns m * kQuadsPerBlock consecutive buckets of one slot (m = 2^log_m per quad):
//   1. quad t turns its chunk into LOCAL suffix sums in place (m - 1 additions, stored back over the buckets);
//   2. a Hillis-Steele suffix scan over the chunk totals in shared memory gives RS_t = sum_{u >= t} S_u (log2 T steps);
//   3. the block's sum of suffix sums is  sum_k R_k(local) + m * sum_{t >= 1} RS_t : quad t starts from 2^log_m * RS_t (t >= 1),
//      adds m of the stored local suffix sums (strided, coalesced) and a shared-memory tree adds the quads up.
// Output per block: its weighted sum with weights 1 .. m T (out_w) and its plain sum RS_0 (out_s); k_reduce_top combines the
// blocks of a slot the same way (suffix scan over the block sums, weight 2^log_u = m T).  Slots with fewer than m T buckets
// share a block (group = quads per slot; the scan and the tree stop at the group boundary).
// (The same scan form with one THREAD per chunk was measured slower than k_reduce at every size:
// profiles/r02c_bucket_slices_and_scan_reduce.md.)
constexpr int kQuadsPerBlock = 64;
constexpr int kQuadThreads = 4 * kQuadsPerBlock;
constexpr int kTopMaxBlocks = kQuadsPerBlock * 64;  // blocks per slot k_reduce_top combines (up to 64 per quad)

// ONE copy of the four-lane addition / doubling per kernel (seven inlined field products each time otherwise)
template <class F>
__device__ __noinline__ QuadPoint<F> quad_add_nl(QuadPoint<F> a, QuadPoint<F> b) { return quad_add(a, b); }
template <class F>
__device__ __noinline__ QuadPoint<F> quad_dbl_nl(QuadPoint<F> a) { return quad_dbl(a); }

template <class F>
PORLA_D QuadPoint<F> quad_from_shared(const XYZZ<F>* p) { return QuadPoint<F>{reinterpret_cast<const F*>(p)[threadIdx.x & 3]}; }
template <class F>
PORLA_D void quad_to_shared(XYZZ<F>* p, const QuadPoint<F>& v) { reinterpret_cast<F*>(p)[threadIdx.x & 3] = v.c; }

// sum of sh[first .. first + count) (count a power of two) into sh[first]; l = this quad's index within the group.
// Every warp of the block must call (barriers); warps whose quads all lie outside a level skip its arithmetic.
template <class F>
PORLA_D void quad_tree_sum(XYZZ<F>* sh, uint32_t q, uint32_t l, uint32_t count) {
    for (uint32_t o = count / 2; o > 0; o >>= 1) {
        const bool act = l < o;
        if (__any_sync(kFullMask, act)) {
            QuadPoint<F> x = QuadPoint<F>::inf(), y = QuadPoint<F>::inf();
            if (act) {
                x = quad_from_shared(&sh[q]);
                y = quad_from_shared(&sh[q + o]);
            }
            x = quad_add_nl(x, y);
            if (act) quad_to_shared(&sh[q], x);
        }
        __syncthreads();
    }
}

// inclusive suffix scan over the group's values (a = this quad's value, also left in sh[q])
template <class F>
PORLA_D QuadPoint<F> quad_suffix_scan(XYZZ<F>* sh, uint32_t q, uint32_t l, uint32_t count, QuadPoint<F> a) {
    quad_to_shared(&sh[q], a);
    __syncthreads();
    for (uint32_t d = 1; d < count; d <<= 1) {
        const bool has = l + d < count;
        QuadPoint<F> b = QuadPoint<F>::inf();
        if (has) b = quad_from_shared(&sh[q + d]);
        __syncthreads();
        a = quad_add_nl(a, b);
        if (has) quad_to_shared(&sh[q], a);
        __syncthreads();
    }
    return a;
}

template <class C>
__global__ void __launch_bounds__(kQuadThreads)
k_reduce_scan(XYZZ<typename C::F>* buckets, uint32_t nb, uint32_t log_m, uint32_t group, uint32_t total_slots,
              XYZZ<typename C::F>* __restrict__ out_w, XYZZ<typename C::F>* __restrict__ out_s) {
    using F = typename C::F;
    using Q = QuadPoint<F>;
    __shared__ XYZZ<F> sh[kQuadsPerBlock];
    const uint32_t m = 1u << log_m;
    const uint32_t q = threadIdx.x >> 2;
    uint32_t slot, blk, blocks_per_slot;
    if (group == (uint32_t)kQuadsPerBlock) {
        blocks_per_slot = (nb >> log_m) / kQuadsPerBlock;
        slot = blockIdx.x / blocks_per_slot;
        blk = blockIdx.x - slot * blocks_per_slot;
    } else {
        blocks_per_slot = 1;
        slot = blockIdx.x * (kQuadsPerBlock / group) + q / group;
        blk = 0;
    }
    const uint32_t l = q & (group - 1);                    // quad within its slot's group
    const bool live = slot < total_slots;
    XYZZ<F>* base = buckets + (size_t)slot * nb + (size_t)blk * ((size_t)group << log_m);
    // 1. local suffix sums of the chunk [l m, (l + 1) m), in place
    XYZZ<F>* p = base + ((size_t)l << log_m);
    Q a = Q::inf(), nxt = Q::inf();
    if (live) {
        a = Q::load_coherent(p + (m - 1));
        if (m > 1) nxt = Q::load_coherent(p + (m - 2));
    }
    for (uint32_t k = m - 1; k-- > 0;) {
        const Q b = nxt;
        if (live && k > 0) nxt = Q::load_coherent(p + (k - 1));       // the next bucket travels while this addition runs
        a = quad_add_nl(a, b);
        if (live) a.store(p + k);
    }
    // 2. inclusive suffix scan of the chunk totals over the group (its first barrier also orders step 1's stores before step 3)
    a = quad_suffix_scan(sh, q, l, group, a);
    if (l == 0 && live) a.store(out_s + (size_t)slot * blocks_per_slot + blk);
    // 3. m * RS_l (l >= 1) + the local suffix sums l, l + group, ...
    Q v = l != 0 ? a : Q::inf();
    for (uint32_t d = 0; d < log_m; d++) v = quad_dbl_nl(v);
    nxt = Q::inf();
    if (live) nxt = Q::load_coherent(base + l);
    for (uint32_t i = 0; i < m; i++) {
        const Q b = nxt;
        if (live && i + 1 < m) nxt = Q::load_coherent(base + l + (size_t)(i + 1) * group);
        v = quad_add_nl(v, b);
    }
    __syncthreads();
    quad_to_shared(&sh[q], v);
    __syncthreads();
    quad_tree_sum(sh, q, l, group);
    if (l == 0 && live) quad_from_shared(&sh[q]).store(out_w + (size_t)slot * blocks_per_slot + blk);
}

// One block per window slot; quad b takes `per` = nblk / 64 consecutive blocks of k_reduce_scan (nblk a power of two; per = 1
// up to 64 blocks) and folds them with running sums -- S' = sum S_j, W' = sum W_j + 2^log_u * sum_j j S_j -- after which the
// quads are combined like the blocks themselves: window sum = sum_b W'_b + 2^(log_u + log2 per) * sum_b b S'_b, the second
// term as the sum of the suffix sums RS_b, b >= 1.
template <class C>
__global__ void __launch_bounds__(kQuadThreads)
k_reduce_top(const XYZZ<typename C::F>* __restrict__ in_w, const XYZZ<typename C::F>* __restrict__ in_s, uint32_t nblk_in,
             uint32_t log_u, XYZZ<typename C::F>* __restrict__ wsum) {
    using F = typename C::F;
    using Q = QuadPoint<F>;
    __shared__ XYZZ<F> sh[kQuadsPerBlock];
    const uint32_t b = threadIdx.x >> 2;
    const uint32_t per = nblk_in > (uint32_t)kQuadsPerBlock ? nblk_in / kQuadsPerBlock : 1u;
    const uint32_t nblk = nblk_in / per;                     // quads at work
    const bool live = b < nblk;
    const size_t at = (size_t)blockIdx.x * nblk_in + (size_t)b * per;
    Q a = Q::inf();                                          // S' of this quad's blocks
    Q wq = Q::inf();                                         // W' of this quad's blocks
    if (per == 1) {
        if (live) {
            a = Q::load(in_s + at);
            wq = Q::load(in_w + at);
        }
    } else {
        Q z = Q::inf();                                      // sum_j j S_j over the quad's blocks (block units)
        for (uint32_t j = per; j-- > 0;) {
            Q s = Q::inf(), w = Q::inf();
            if (live) {
                s = Q::load(in_s + at + j);
                w = Q::load(in_w + at + j);
            }
            a = quad_add_nl(a, s);
            wq = quad_add_nl(wq, w);
            if (j != 0) z = quad_add_nl(z, a);
        }
        for (uint32_t d = 0; d < log_u; d++) z = quad_dbl_nl(z);
        wq = quad_add_nl(wq, z);
        for (uint32_t q = per; q > 1; q >>= 1) log_u++;      // a quad now stands for `per` blocks
    }
    a = quad_suffix_scan(sh, b, b, nblk, a);                // quads >= nblk hold infinity and stay out of it
    Q v = (b != 0 && live) ? a : Q::inf();
    for (uint32_t d = 0; d < log_u; d++) v = quad_dbl_nl(v);
    v = quad_add_nl(v, wq);
    __syncthreads();
    quad_to_shared(&sh[b], v);
    __syncthreads();
    quad_tree_sum(sh, b, b, nblk);
    if (b == 0) quad_from_shared(&sh[0]).store(wsum + blockIdx.x);
}

// ---------------------------------------------------------------------------- window sums
// Sums the per-block partials of one window slot with a block-wide tree (replaces a serial loop
// in the finaliser): wsum[slot] = sum_k partials[slot*count + k].
template <class C>
__global__ void __launch_bounds__(kRedThreads)
k_window_sums(const XYZZ<typename C::FC>* __restrict__ partials, uint32_t count,
              XYZZ<typename C::FC>* __restrict__ wsum) {
    using F = typename C::FC;
    __shared__ XYZZ<F> sh[kRedThreads];
    const XYZZ<F>* p = partials + (size_t)blockIdx.x * count;
    XYZZ<F> acc = XYZZ<F>::inf();
    for (uint32_t k = threadIdx.x; k < count; k += kRedThreads) acc.add(ld16(p + k));
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int o = kRedThreads / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
            XYZZ<F> a = sh[threadIdx.x];
            a.add(sh[threadIdx.x + o]);
            sh[threadIdx.x] = a;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) st16(wsum + blockIdx.x, sh[0]);
}

// ---------------------------------------------------------------------------- finalisation
// One thread per MSM: Horner over the window sums (c doublings each; doubling infinity is free so
// leading empty windows cost nothing), normalise to affine, serialise.  out_fmt: kPointBE64 / kPointLE64 external bytes
// (canonical, not Montgomery); out_xyzz (optional) receives the un-normalised sum for multi-GPU
// combination.
template <class C>
__global__ void __launch_bounds__(32)
k_finalize(const XYZZ<typename C::FC>* __restrict__ wsums, uint32_t nbatch, int nwin, int c, int out_fmt,
           uint8_t* __restrict__ out, XYZZ<typename C::FC>* __restrict__ out_xyzz) {
    using F = typename C::FC;
    // one thread per MSM (a batch of MSMs fills warps; a single MSM is one serial chain)
    const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= nbatch) return;
    const XYZZ<F>* ws = wsums + (size_t)m * nwin;
    XYZZ<F> r = XYZZ<F>::inf();
    for (int w = nwin - 1; w >= 0; w--) {
        if (!r.is_inf())
            for (int k = 0; k < c; k++) r = r.dbl();
        r.add(ld16(ws + w));
    }
    if (out_xyzz) st16(out_xyzz + m, r);
    if (out) {
        Affine<F> a = r.to_affine();
        F x = a.x.from_internal(), y = a.y.from_internal();
        store_u256(out, 2 * (size_t)m, out_fmt == kPointBE64, x.v);
        store_u256(out, 2 * (size_t)m + 1, out_fmt == kPointBE64, y.v);
    }
}

// Sum `count` XYZZ partial results per MSM (multi-GPU combine) and serialise.
template <class C>
__global__ void k_combine(const XYZZ<typename C::FC>* __restrict__ parts, uint32_t count,
                          uint32_t nbatch, int out_fmt, uint8_t* __restrict__ out) {
    using F = typename C::FC;
    uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= nbatch) return;
    XYZZ<F> r = XYZZ<F>::inf();
    for (uint32_t k = 0; k < count; k++) r.add(ld16(parts + (size_t)k * nbatch + m));
    Affine<F> a = r.to_affine();
    F x = a.x.from_internal(), y = a.y.from_internal();
    store_u256(out, 2 * (size_t)m, out_fmt == kPointBE64, x.v);
    store_u256(out, 2 * (size_t)m + 1, out_fmt == kPointBE64, y.v);
}

// ---------------------------------------------------------------------------- elementwise ops
// Batched single-point kernels (SURVEY.md 8(f)1: the "FFT in the exponent" butterflies issue
// these through mult_point/add_point/neg_point, main.go:196-222) and test hooks.
// out[i] = k_i * P_i, scalars 32-byte records, plain double-and-add.
template <class C>
__global__ void __launch_bounds__(128)
k_scalar_mul(const Affine<typename C::FC>* __restrict__ points, uint32_t npoints,
             const uint8_t* __restrict__ scalars, int big_endian, uint32_t n,
             Affine<typename C::FC>* __restrict__ out) {
    using F = typename C::FC;
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t s[8];
    load_u256(scalars, i, big_endian, s);
    reduce_scalar<C>(s);
    Affine<F> p = ld16(points + (npoints == 1 ? 0 : i));
    XYZZ<F> r = XYZZ<F>::inf();
    if (!p.is_inf()) {
        int top = 255;
        while (top >= 0 && !((s[top >> 5] >> (top & 31)) & 1u)) top--;
        for (int b = top; b >= 0; b--) {
            r = r.dbl();
            if ((s[b >> 5] >> (b & 31)) & 1u) r.madd(p);
        }
    }
    st16(out + i, r.to_affine());
}

// One radix-2 stage of Porla's "FFT in the exponent" (CRebuild / mix: /root/reference/porla/Server/
// Server.hpp:1548-1687 and :1209-1328, Client.hpp:921-976): for every j < m/2 and k = j, j + m, ... < n
//     t = w_j * P[k + m/2];   P[k] <- P[k] + t;   P[k + m/2] <- P[k] - t
// which the reference issues as mult_point + add_point + neg_point + add_point per butterfly
// (main.go:196-222) or secp256k1_ecmult + 2 gej_add_var in IPA mode.  One thread per butterfly, in
// place on the resident affine table; both outputs share one field inversion.  flags[] (1 =
// infinity) is rewritten so that MSMs over the table keep skipping infinities.
template <class C, class F>
__global__ void __launch_bounds__(128)
k_butterfly(Affine<F>* __restrict__ pts, uint8_t* __restrict__ flags, uint32_t n, uint32_t m,
            const uint8_t* __restrict__ twiddles, int big_endian) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t m2 = m >> 1;
    if (b >= n / 2) return;
    const uint32_t j = b % m2, k = (b / m2) * m + j;
    uint32_t s[8];
    load_u256(twiddles, j, big_endian, s);
    reduce_scalar<C>(s);
    const Affine<F> a0 = ld16(pts + k), a1 = ld16(pts + k + m2);
    XYZZ<F> t = XYZZ<F>::inf();
    // w = k1 + k2 lambda: joint double-and-add over (P, phi(P), P + phi(P)), 127 (BN254) or 128 (secp256k1) doublings
    // instead of 254 or 256.
    // Every lane of the warp adds an AFFINE operand chosen by its two bits (infinity for 00), so the warp
    // executes one doubling and one mixed addition per bit whatever the lanes' digits are.
    if (!a1.is_inf()) {
        uint32_t k1[4], k2[4], n1, n2;
        glv_split<C>(s, k1, k2, n1, n2);
        Affine<F> tab[3];
        tab[0] = a1;
        if (n1) tab[0].y = tab[0].y.neg();
        F beta;
#pragma unroll
        for (int q = 0; q < 8; q++) beta.v[q] = C::glv_beta_mont(q);
        tab[1].x = a1.x * beta;
        tab[1].y = n2 ? a1.y.neg() : a1.y;
        XYZZ<F> both = XYZZ<F>::from_affine(tab[0]);
        both.madd(tab[1]);
        tab[2] = both.to_affine();          // (+-1 +- lambda) P is never infinity: lambda != +-1
        int top = 127;
        while (top >= 0 && !(((k1[top >> 5] | k2[top >> 5]) >> (top & 31)) & 1u)) top--;
#pragma unroll 1
        for (int i = top; i >= 0; i--) {
            t = t.dbl();
            const uint32_t b = ((k1[i >> 5] >> (i & 31)) & 1u) | (((k2[i >> 5] >> (i & 31)) & 1u) << 1);
            Affine<F> q = Affine<F>::inf();
            if (b == 1) q = tab[0];
            else if (b == 2) q = tab[1];
            else if (b == 3) q = tab[2];
            t.madd(q);
        }
    }
    XYZZ<F> r0 = t, r1 = t.neg();
    r0.madd(a0);
    r1.madd(a0);
    // joint normalisation: 1/zzz0 and 1/zzz1 from one inversion of their product
    Affine<F> o0 = Affine<F>::inf(), o1 = Affine<F>::inf();
    if (r0.is_inf() || r1.is_inf()) {
        o0 = r0.to_affine();
        o1 = r1.to_affine();
    } else {
        F inv = (r0.zzz * r1.zzz).inverse();
        F i0 = inv * r1.zzz, i1 = inv * r0.zzz;
        F t0 = r0.zz * i0, t1 = r1.zz * i1;   // 1/zz = (zz/zzz)^2
        o0.x = r0.x * t0.sqr();
        o0.y = r0.y * i0;
        o1.x = r1.x * t1.sqr();
        o1.y = r1.y * i1;
    }
    st16(pts + k, o0);
    st16(pts + k + m2, o1);
    if (flags) {
        flags[k] = o0.is_inf() ? 1 : 0;
        flags[k + m2] = o1.is_inf() ? 1 : 0;
    }
}

// The same stage with FOUR lanes per butterfly (quad.cuh), for stages of few butterflies where the 127 dependent doublings and
// additions are pure latency (Porla's rebuild of 1024 blocks: 512 butterflies per stage on a 148-SM part).
// Differences from k_butterfly besides the lane layout:
//   - joint 2-bit windows over the halves of w = k1 + k2 lambda: a table of the 15 combinations d1 (+-P) + d2 (+-phi(P)),
//     0 <= d1, d2 <= 3, kept in shared memory in XYZZ form (the four-lane addition takes general operands, so nothing is
//     normalised: A, 2A, 3A, their images under phi -- one product by beta each -- and nine additions), then 64 steps of two
//     doublings and ONE addition instead of 127 steps of a doubling and an addition;
//   - the loop bound is the warp's largest digit count, so that all lanes shuffle together;
//   - the joint normalisation of the two outputs is done by the quad's first lane on the gathered points.
constexpr int kBflyQuadThreads = 64;     // 16 quads x 16 table entries x 128 B = 32 KB of shared memory
template <class C>
__global__ void __launch_bounds__(kBflyQuadThreads)
k_butterfly_quad(Affine<typename C::F>* __restrict__ pts, uint8_t* __restrict__ flags, uint32_t n, uint32_t m,
                 const uint8_t* __restrict__ twiddles, int big_endian) {
    using F = typename C::F;
    using Q = QuadPoint<F>;
    __shared__ F tab[kBflyQuadThreads / 4][16][4];
    const uint32_t b = (blockIdx.x * blockDim.x + threadIdx.x) >> 2, role = threadIdx.x & 3, ql = threadIdx.x >> 2;
    const uint32_t m2 = m >> 1;
    const bool live = b < n / 2;
    const uint32_t bb = live ? b : 0u;
    const uint32_t j = bb % m2, k = (bb / m2) * m + j;
    uint32_t k1[4], k2[4], n1, n2;
    glv_scalar<C>(twiddles, j, big_endian, k1, k2, n1, n2);
    Q a1 = Q::load_affine(pts + k + m2, false);
    if (!live) a1 = Q::inf();
    {
        F beta;
#pragma unroll
        for (int q = 0; q < 8; q++) beta.v[q] = C::glv_beta_mont(q);
        Q mult[3];
        mult[0] = a1;
        mult[1] = quad_dbl_nl(a1);
        mult[2] = quad_add_nl(mult[1], a1);
#pragma unroll 1
        for (int d = 1; d <= 3; d++) {
            Q e1 = mult[d - 1], e2 = mult[d - 1];
            const F bx = e2.c * beta;                      // phi: X -> beta X (lane 0)
            if (role == 0) e2.c = bx;
            if (role == 1) {
                if (n1) e1.c = e1.c.neg();
                if (n2) e2.c = e2.c.neg();
            }
            tab[ql][d][role] = e1.c;                       // d (+-P)
            tab[ql][4 * d][role] = e2.c;                   // d (+-phi(P))
        }
        __syncwarp();
#pragma unroll 1
        for (int d2 = 1; d2 <= 3; d2++) {
#pragma unroll 1
            for (int d1 = 1; d1 <= 3; d1++) {
                const Q x = quad_add_nl(Q{tab[ql][d1][role]}, Q{tab[ql][4 * d2][role]});
                tab[ql][d1 + 4 * d2][role] = x.c;
            }
        }
        __syncwarp();
    }
    int top = 63;                                          // digit positions: bits 2 i, 2 i + 1 of k1 and of k2
    while (top >= 0 && !(((k1[top >> 4] | k2[top >> 4]) >> ((top & 15) * 2)) & 3u)) top--;
    if (!live) top = -1;
    top = __reduce_max_sync(kFullMask, top);
    Q t = Q::inf();
#pragma unroll 1
    for (int i = top; i >= 0; i--) {
        t = quad_dbl_nl(t);
        t = quad_dbl_nl(t);
        const uint32_t e = ((k1[i >> 4] >> ((i & 15) * 2)) & 3u) | (((k2[i >> 4] >> ((i & 15) * 2)) & 3u) << 2);
        Q q = Q::inf();
        if (e != 0) q.c = tab[ql][e][role];
        t = quad_add_nl(t, q);
    }
    Q a0 = Q::load_affine(pts + k, false);
    if (!live) a0 = Q::inf();
    Q tn = t;
    if (role == 1) tn.c = tn.c.neg();
    const XYZZ<F> r0 = quad_add_nl(t, a0).gather(), r1 = quad_add_nl(tn, a0).gather();
    if (!live || role != 0) return;
    Affine<F> o0 = Affine<F>::inf(), o1 = Affine<F>::inf();
    if (r0.is_inf() || r1.is_inf()) {
        o0 = r0.to_affine();
        o1 = r1.to_affine();
    } else {
        F inv = (r0.zzz * r1.zzz).inverse();
        F i0 = inv * r1.zzz, i1 = inv * r0.zzz;
        F t0 = r0.zz * i0, t1 = r1.zz * i1;   // 1/zz = (zz/zzz)^2
        o0.x = r0.x * t0.sqr();
        o0.y = r0.y * i0;
        o1.x = r1.x * t1.sqr();
        o1.y = r1.y * i1;
    }
    st16(pts + k, o0);
    st16(pts + k + m2, o1);
    if (flags) {
        flags[k] = o0.is_inf() ? 1 : 0;
        flags[k + m2] = o1.is_inf() ? 1 : 0;
    }
}

// ---- Server::align_MAC scalar preparation (/root/reference/porla/Server/Server.hpp:531-540, KZG branch)
// rem = a mod m for a 512-bit a (16 LE limbs) and a 256-bit m: restoring shift-subtract, one bit per step.
// The values are touched once and the kernel is a few hundred kilobytes of traffic per launch; no attempt
// at a word-wise division is made.
PORLA_D void mod512(const uint32_t* a, const uint32_t* m, uint32_t* rem) {
#pragma unroll
    for (int k = 0; k < 8; k++) rem[k] = 0;
    for (int bit = 511; bit >= 0; bit--) {
        uint32_t top = rem[7] >> 31;
#pragma unroll
        for (int k = 7; k > 0; k--) rem[k] = (rem[k] << 1) | (rem[k - 1] >> 31);
        rem[0] = (rem[0] << 1) | ((a[bit >> 5] >> (bit & 31)) & 1u);
        uint32_t t[8];
        uint32_t borrow = sub256(t, rem, m);
        if (top | (borrow ^ 1u)) {   // 2 rem + bit >= m
#pragma unroll
            for (int k = 0; k < 8; k++) rem[k] = t[k];
        }
    }
}

// One thread per chunk:  mod = A % PRIME_MODULUS;  c = (mod - A) % r;  A <- mod;  c -> 32-byte big-endian
// scalar for the commitment.  PRIME_MODULUS = 207 * 2^248 + 1 (utils.h:40), r = C's group order: BN254's in KZG mode
// (utils.h:37), secp256k1's n in IPA mode (GROUP_ORDER, utils.h:32).
template <class C>
__global__ void __launch_bounds__(128)
k_align_scalars(uint32_t* __restrict__ data, uint32_t total, uint8_t* __restrict__ scalars_be) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    constexpr uint32_t kPrime[8] = {0x00000001u, 0u, 0u, 0u, 0u, 0u, 0u, 0xcf000000u};
    uint32_t a[16], pm[8], ord[8], rem[8], d[16], t[8], c[8];
    uint4* src = reinterpret_cast<uint4*>(data + (size_t)i * 16);
#pragma unroll
    for (int k = 0; k < 4; k++) {
        uint4 v = src[k];
        a[4 * k] = v.x; a[4 * k + 1] = v.y; a[4 * k + 2] = v.z; a[4 * k + 3] = v.w;
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
        pm[k] = kPrime[k];
        ord[k] = C::order(k);
    }
    mod512(a, pm, rem);
    // d = A - mod  (a multiple of PRIME_MODULUS, non-negative)
    uint32_t borrow = 0;
#pragma unroll
    for (int k = 0; k < 16; k++) {
        uint32_t sub = k < 8 ? rem[k] : 0u;
        uint64_t v = (uint64_t)a[k] - sub - borrow;
        d[k] = (uint32_t)v;
        borrow = (uint32_t)(v >> 63);
    }
    mod512(d, ord, t);
    // c = (-(A - mod)) mod r
    bool zero = true;
#pragma unroll
    for (int k = 0; k < 8; k++) zero = zero && t[k] == 0;
    sub256(c, ord, t);
#pragma unroll
    for (int k = 0; k < 8; k++) c[k] = zero ? 0u : c[k];
    store_u256(scalars_be, i, 1, c);
#pragma unroll
    for (int k = 0; k < 4; k++)
        src[k] = k < 2 ? make_uint4(rem[4 * k], rem[4 * k + 1], rem[4 * k + 2], rem[4 * k + 3]) : make_uint4(0u, 0u, 0u, 0u);
}

// ---- Server::audit block aggregation + alignment (/root/reference/porla/Server/Server.hpp:790-828, 531-540; SURVEY 8(f)4)
// rem = a mod m for an a of LIMBS 32-bit limbs and a 256-bit m (restoring shift-subtract, as mod512).
template <int LIMBS>
PORLA_D void mod_wide(const uint32_t* a, const uint32_t* m, uint32_t* rem) {
#pragma unroll
    for (int k = 0; k < 8; k++) rem[k] = 0;
    for (int bit = LIMBS * 32 - 1; bit >= 0; bit--) {
        uint32_t top = rem[7] >> 31;
#pragma unroll
        for (int k = 7; k > 0; k--) rem[k] = (rem[k] << 1) | (rem[k - 1] >> 31);
        rem[0] = (rem[0] << 1) | ((a[bit >> 5] >> (bit & 31)) & 1u);
        uint32_t t[8];
        uint32_t borrow = sub256(t, rem, m);
        if (top | (borrow ^ 1u)) {
#pragma unroll
            for (int k = 0; k < 8; k++) rem[k] = t[k];
        }
    }
}

// Block j of the grid owns chunk j:  B = sum_i coefs[i] * blocks[i][j]  (plain integers: coefficients below 2^31,
// chunks of 16 LE limbs, at most 2^24 blocks, so B < 2^567 fits kAggLimbs limbs), thread t takes the blocks
// i = t, t + 128, ...; the partial sums meet in a shared-memory tree.  Thread 0 then applies align_MAC's
// arithmetic:  mod = B % PRIME_MODULUS,  c = (mod - B) % r,  and emits both as 32-byte big-endian scalars.
constexpr int kAggLimbs = 18;
constexpr int kAggThreads = 128;
template <class C>
__global__ void __launch_bounds__(kAggThreads)
k_audit_aggregate(const uint32_t* __restrict__ coefs, const uint32_t* __restrict__ blocks, uint32_t n, uint32_t chunks,
                  uint8_t* __restrict__ b_mod_be, uint8_t* __restrict__ c_be) {
    __shared__ uint32_t sh[kAggThreads][kAggLimbs + 1];   // +1: bank spread
    const uint32_t j = blockIdx.x;
    uint32_t acc[kAggLimbs];
#pragma unroll
    for (int k = 0; k < kAggLimbs; k++) acc[k] = 0;
    for (uint32_t i = threadIdx.x; i < n; i += kAggThreads) {
        const uint32_t cf = __ldg(coefs + i);
        const uint4* src = reinterpret_cast<const uint4*>(blocks + ((size_t)i * chunks + j) * 16);
        uint32_t a[16];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            uint4 v = __ldg(src + k);
            a[4 * k] = v.x; a[4 * k + 1] = v.y; a[4 * k + 2] = v.z; a[4 * k + 3] = v.w;
        }
        uint64_t carry = 0;
#pragma unroll
        for (int k = 0; k < 16; k++) {
            uint64_t v = (uint64_t)a[k] * cf + acc[k] + carry;
            acc[k] = (uint32_t)v;
            carry = v >> 32;
        }
#pragma unroll
        for (int k = 16; k < kAggLimbs; k++) {
            uint64_t v = (uint64_t)acc[k] + carry;
            acc[k] = (uint32_t)v;
            carry = v >> 32;
        }
    }
#pragma unroll
    for (int k = 0; k < kAggLimbs; k++) sh[threadIdx.x][k] = acc[k];
    __syncthreads();
    for (int o = kAggThreads / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
            uint32_t carry = 0;
#pragma unroll
            for (int k = 0; k < kAggLimbs; k++) {
                uint64_t v = (uint64_t)sh[threadIdx.x][k] + sh[threadIdx.x + o][k] + carry;
                sh[threadIdx.x][k] = (uint32_t)v;
                carry = (uint32_t)(v >> 32);
            }
        }
        __syncthreads();
    }
    if (threadIdx.x != 0) return;
    constexpr uint32_t kPrime[8] = {0x00000001u, 0u, 0u, 0u, 0u, 0u, 0u, 0xcf000000u};
    uint32_t B[kAggLimbs], pm[8], ord[8], rem[8], d[kAggLimbs], t[8], c[8];
#pragma unroll
    for (int k = 0; k < kAggLimbs; k++) B[k] = sh[0][k];
#pragma unroll
    for (int k = 0; k < 8; k++) {
        pm[k] = kPrime[k];
        ord[k] = C::order(k);
    }
    mod_wide<kAggLimbs>(B, pm, rem);
    uint32_t borrow = 0;   // d = B - mod, a non-negative multiple of PRIME_MODULUS
#pragma unroll
    for (int k = 0; k < kAggLimbs; k++) {
        uint32_t sub = k < 8 ? rem[k] : 0u;
        uint64_t v = (uint64_t)B[k] - sub - borrow;
        d[k] = (uint32_t)v;
        borrow = (uint32_t)(v >> 63);
    }
    mod_wide<kAggLimbs>(d, ord, t);
    bool zero = true;
#pragma unroll
    for (int k = 0; k < 8; k++) zero = zero && t[k] == 0;
    sub256(c, ord, t);   // c = (-(B - mod)) mod r
#pragma unroll
    for (int k = 0; k < 8; k++) c[k] = zero ? 0u : c[k];
    store_u256(c_be, j, 1, c);
    store_u256(b_mod_be, j, 1, rem);
}

// ---- data side of the FFT (CRebuild / mix on the blocks themselves; /root/reference/porla/Server/Server.hpp:1582-1588,
// :1240-1246; SURVEY 8(f)4): for every butterfly (k, k + m/2) of a stage and every chunk p
//     t = v_j * X[k + m/2][p];   X[k][p] = (u + t) % LCM;   X[k + m/2][p] = (u - t) % LCM      (u = X[k][p])
// on 512-bit chunks (16 LE limbs, values below LCM < 2^511, utils.h:42-43) with a 256-bit twiddle.  One thread per
// (butterfly, chunk); t is reduced with Barrett's method (mu = floor(2^1022 / LCM) computed once on the host), the sum
// and the difference then need one conditional correction each.  64 B read and written per chunk: HBM-bound.
struct DataFftParams {
    uint32_t lcm[16];
    uint32_t mu[17];      // floor(2^1022 / LCM), < 2^513
};

// r = a - b on N limbs, returns the borrow
template <int N>
PORLA_D uint32_t sub_limbs(uint32_t* r, const uint32_t* a, const uint32_t* b) {
    uint32_t borrow = 0;
#pragma unroll
    for (int i = 0; i < N; i++) {
        uint64_t d = (uint64_t)a[i] - b[i] - borrow;
        r[i] = (uint32_t)d;
        borrow = (uint32_t)(d >> 63);
    }
    return borrow;
}

static __global__ void __launch_bounds__(128)
k_data_butterfly(uint32_t* __restrict__ blocks, uint32_t n_blocks, uint32_t chunks, uint32_t m,
                 const uint8_t* __restrict__ twiddles_le32, DataFftParams prm) {
    const uint64_t gid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t m2 = m >> 1;
    const uint64_t total = (uint64_t)(n_blocks / 2) * chunks;
    if (gid >= total) return;
    const uint32_t bfly = (uint32_t)(gid / chunks), p = (uint32_t)(gid - (uint64_t)bfly * chunks);
    const uint32_t j = bfly % m2, k = (bfly / m2) * m + j;
    uint4* pu = reinterpret_cast<uint4*>(blocks + ((size_t)k * chunks + p) * 16);
    uint4* px = reinterpret_cast<uint4*>(blocks + ((size_t)(k + m2) * chunks + p) * 16);
    uint32_t u[16], x[16], v[8];
#pragma unroll
    for (int q = 0; q < 4; q++) {
        uint4 a = pu[q], b = px[q];
        u[4 * q] = a.x; u[4 * q + 1] = a.y; u[4 * q + 2] = a.z; u[4 * q + 3] = a.w;
        x[4 * q] = b.x; x[4 * q + 1] = b.y; x[4 * q + 2] = b.z; x[4 * q + 3] = b.w;
    }
    load_u256(twiddles_le32, j, 0, v);
    // t = v * x  (24 limbs, < 2^767)
    uint32_t t[25];
    mul_limbs<8, 16, 24>(v, x, t);
    t[24] = 0;
    // Barrett: q1 = t >> 510, q3 ~ (q1 * mu) >> 512, r = t - q3 * LCM  (0 <= r < 4 LCM), all mod 2^544
    uint32_t q1[9];
#pragma unroll
    for (int i = 0; i < 9; i++) q1[i] = __funnelshift_r(t[15 + i], t[16 + i], 30);
    // q3 = (q1 * mu) >> 512 from the partial products at limb 14 and above only: the dropped ones (i + j <= 13, ninety
    // products below 2^480 each) change q1 * mu by less than 2^487, so q3 is at most one too small and r stays below 4 LCM
    uint32_t q2h[12];   // limbs 14 .. 25 of the product
#pragma unroll
    for (int i = 0; i < 12; i++) q2h[i] = 0;
#pragma unroll
    for (int i = 0; i < 9; i++) {
        uint64_t carry = 0;
#pragma unroll
        for (int j = 0; j < 17; j++) {
            if (i + j >= 14) {
                uint64_t pv = (uint64_t)q1[i] * prm.mu[j] + q2h[i + j - 14] + carry;
                q2h[i + j - 14] = (uint32_t)pv;
                carry = pv >> 32;
            }
        }
        q2h[i + 17 - 14] = (uint32_t)carry;
    }
    uint32_t q3[10];
#pragma unroll
    for (int i = 0; i < 10; i++) q3[i] = q2h[2 + i];
    uint32_t qm[17], r[17];
    mul_limbs<10, 16, 17>(q3, prm.lcm, qm);
    sub_limbs<17>(r, t, qm);
    uint32_t lc[17];
#pragma unroll
    for (int i = 0; i < 16; i++) lc[i] = prm.lcm[i];
    lc[16] = 0;
#pragma unroll 1
    for (int it = 0; it < 3; it++) {
        uint32_t d[17];
        if (!sub_limbs<17>(d, r, lc)) {
#pragma unroll
            for (int i = 0; i < 17; i++) r[i] = d[i];
        }
    }
    // sum and difference mod LCM
    uint32_t s0[17], s1[17], uu[17];
#pragma unroll
    for (int i = 0; i < 16; i++) uu[i] = u[i];
    uu[16] = 0;
    uint32_t carry = 0;
#pragma unroll
    for (int i = 0; i < 17; i++) {
        uint64_t a = (uint64_t)uu[i] + r[i] + carry;
        s0[i] = (uint32_t)a;
        carry = (uint32_t)(a >> 32);
    }
    {
        uint32_t d[17];
        if (!sub_limbs<17>(d, s0, lc)) {
#pragma unroll
            for (int i = 0; i < 17; i++) s0[i] = d[i];
        }
    }
    if (sub_limbs<17>(s1, uu, r)) {   // u < t': add LCM back
        carry = 0;
#pragma unroll
        for (int i = 0; i < 17; i++) {
            uint64_t a = (uint64_t)s1[i] + lc[i] + carry;
            s1[i] = (uint32_t)a;
            carry = (uint32_t)(a >> 32);
        }
    }
#pragma unroll
    for (int q = 0; q < 4; q++) {
        pu[q] = make_uint4(s0[4 * q], s0[4 * q + 1], s0[4 * q + 2], s0[4 * q + 3]);
        px[q] = make_uint4(s1[4 * q], s1[4 * q + 1], s1[4 * q + 2], s1[4 * q + 3]);
    }
}

// out[i] = a[i] + b[i]
template <class C>
__global__ void k_point_add(const Affine<typename C::FC>* __restrict__ a,
                            const Affine<typename C::FC>* __restrict__ b, uint32_t n,
                            Affine<typename C::FC>* __restrict__ out) {
    using F = typename C::FC;
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    XYZZ<F> r = XYZZ<F>::from_affine(ld16(a + i));
    r.madd(ld16(b + i));
    st16(out + i, r.to_affine());
}

// out[i] = a[i] * b[i] on raw field elements (internal form) -- unit-test hook for the PTX path
// op 0: a*b   1: a^2   2: a*b + b*(a+b) through the fused product-sum
template <class C>
__global__ void k_field_mul(const typename C::F* __restrict__ a, const typename C::F* __restrict__ b,
                            uint32_t n, int op, typename C::F* __restrict__ out) {
    using F = typename C::F;
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (op == 0) out[i] = a[i] * b[i];
    else if (op == 1) out[i] = a[i].sqr();
    else out[i] = F::mul2add(a[i], b[i], b[i], a[i] + b[i]);
}

}  // namespace porla
