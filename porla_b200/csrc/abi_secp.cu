// secp256k1 (Porla IPA mode) boundary: a drop-in for the static secp256k1_ecmult_multi_var of
// /root/reference/porla/Utils/secp256k1_lib/ecmult_impl.h:814-860 operating on the reference's
// own struct layouts (field_5x52.h:12-21, group.h:13-28, scalar_4x64.h:13-15), plus the SEC1
// serialiser (eckey_impl.h:36-52) used as the parity format.  Conversion rules: SURVEY.md App. E.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/porla_multiexp.h"
#include "host_bn254.hpp"
#include "msm.h"
#include "staging.h"

using namespace porla;

namespace {

typedef unsigned __int128 u128;

// secp256k1_fe (5x52, any magnitude) -> canonical 8x32 LE limbs below p
// (the effect of secp256k1_fe_normalize_var, field_5x52_impl.h:128-170, then fe_get_b32 :344-381)
void fe_to_canonical(const porla_secp256k1_fe* a, uint32_t out[8]) {
    uint32_t w[11] = {0};  // 352 bits are plenty: sum of n[i] << 52i < 2^273
    for (int i = 0; i < 5; i++) {
        int bit = 52 * i;
        u128 v = (u128)a->n[i] << (bit & 31);
        int k = bit >> 5;
        uint64_t carry = 0;
        for (int j = 0; j < 4 && k + j < 11; j++) {
            uint64_t s = (uint64_t)w[k + j] + (uint32_t)(v >> (32 * j)) + carry;
            w[k + j] = (uint32_t)s;
            carry = s >> 32;
        }
        for (int j = k + 4; carry && j < 11; j++) {
            uint64_t s = (uint64_t)w[j] + carry;
            w[j] = (uint32_t)s;
            carry = s >> 32;
        }
    }
    // fold limbs 8.. : 2^256 = 2^32 + 977 (mod p), twice
    for (int round = 0; round < 3; round++) {
        uint64_t hi = (uint64_t)w[8] | ((uint64_t)w[9] << 32);
        if (w[10]) { fprintf(stderr, "[libmultiexp/porla_b200] FATAL: secp256k1_fe magnitude too large\n"); abort(); }
        if (!hi) break;
        w[8] = w[9] = 0;
        u128 add0 = (u128)hi * 977u;          // at limb 0
        u128 add1 = (u128)hi;                 // at limb 1
        uint64_t carry = 0;
        for (int j = 0; j < 10; j++) {
            u128 s = (u128)w[j] + carry;
            if (j < 4) s += (uint32_t)(add0 >> (32 * j));
            if (j >= 1 && j < 4) s += (uint32_t)(add1 >> (32 * (j - 1)));
            w[j] = (uint32_t)s;
            carry = (uint64_t)(s >> 32);
        }
    }
    memcpy(out, w, 32);
    host::reduce_canonical<SecpFp>(out);
}

// canonical 8x32 -> 5x52 (fe_set_b32 layout, field_5x52_impl.h:294-341)
void canonical_to_fe(const uint32_t in[8], porla_secp256k1_fe* r) {
    uint64_t q[4];
    for (int i = 0; i < 4; i++) q[i] = (uint64_t)in[2 * i] | ((uint64_t)in[2 * i + 1] << 32);
    const uint64_t M = 0xFFFFFFFFFFFFFull;
    r->n[0] = q[0] & M;
    r->n[1] = ((q[0] >> 52) | (q[1] << 12)) & M;
    r->n[2] = ((q[1] >> 40) | (q[2] << 24)) & M;
    r->n[3] = ((q[2] >> 28) | (q[3] << 36)) & M;
    r->n[4] = q[3] >> 16;
}

void gej_set_infinity(porla_secp256k1_gej* r) {
    memset(r, 0, sizeof(*r));
    r->infinity = 1;
}

using SF = host::Fp64<host::SecpFq64Params>;

// secp256k1_gej (Jacobian, any z, any field magnitude) -> canonical affine x = X / Z^2, y = Y / Z^3 (no inversion when
// Z = 1); infinity -> Affine::inf()
Affine<SF> gej_to_affine(const porla_secp256k1_gej* a) {
    if (a->infinity) return Affine<SF>::inf();
    uint32_t x[8], y[8], z[8];
    fe_to_canonical(&a->x, x);
    fe_to_canonical(&a->y, y);
    fe_to_canonical(&a->z, z);
    Affine<SF> r;
    SF zf;
    memcpy(r.x.v, x, 32);
    memcpy(r.y.v, y, 32);
    memcpy(zf.v, z, 32);
    if (zf != SF::one()) {
        const SF zi = zf.inverse(), zi2 = zi.sqr();
        r.x = r.x * zi2;
        r.y = r.y * zi2 * zi;
    }
    return r;
}

// 64 bytes of canonical LE affine x || y (all zero: infinity) -> gej with z = 1, or infinity as gej_set_infinity writes it
void gej_from_le64(const uint8_t* b, porla_secp256k1_gej* r) {
    uint32_t xy[16];
    memcpy(xy, b, 64);
    bool inf = true;
    for (int i = 0; i < 16; i++) inf = inf && xy[i] == 0;
    if (inf) {
        gej_set_infinity(r);
        return;
    }
    canonical_to_fe(xy, &r->x);
    canonical_to_fe(xy + 8, &r->y);
    memset(&r->z, 0, sizeof(r->z));
    r->z.n[0] = 1;
    r->infinity = 0;
}

void gej_batch_from_le64(const uint8_t* b, size_t n, porla_secp256k1_gej* r) {
    for (size_t i = 0; i < n; i++) gej_from_le64(b + 64 * i, r + i);
}

const uint8_t kGenLE[64] = {
    // x, y of G as 8 LE 32-bit limbs each (little-endian bytes)
    0x98, 0x17, 0xF8, 0x16, 0x5B, 0x81, 0xF2, 0x59, 0xD9, 0x28, 0xCE, 0x2D, 0xDB, 0xFC, 0x9B, 0x02,
    0x07, 0x0B, 0x87, 0xCE, 0x95, 0x62, 0xA0, 0x55, 0xAC, 0xBB, 0xDC, 0xF9, 0x7E, 0x66, 0xBE, 0x79,
    0xB8, 0xD4, 0x10, 0xFB, 0x8F, 0xD0, 0x47, 0x9C, 0x19, 0x54, 0x85, 0xA6, 0x48, 0xB4, 0x17, 0xFD,
    0xA8, 0x08, 0x11, 0x0E, 0xFC, 0xFB, 0xA4, 0x5D, 0x65, 0xC4, 0xA3, 0x26, 0x77, 0xDA, 0x3A, 0x48};

template <class C>
void point_add_host(const uint8_t* a, const uint8_t* b, int64_t n, int fmt, uint8_t* out) {
    using F = typename C::F;
    for (int64_t i = 0; i < n; i++) {
        Affine<F> p, q;
        const uint8_t* pa = a + 64 * i;
        const uint8_t* pb = b + 64 * i;
        auto load = [&](const uint8_t* s, F* x) {
            if (fmt == PORLA_POINT_BE64) host::be32_to_limbs(s, x->v);
            else memcpy(x->v, s, 32);
            host::reduce_canonical<F>(x->v);
            *x = x->to_internal();
        };
        load(pa, &p.x); load(pa + 32, &p.y); load(pb, &q.x); load(pb + 32, &q.y);
        XYZZ<F> r = XYZZ<F>::from_affine(p);
        r.madd(q);
        Affine<F> s = r.to_affine();
        F x = s.x.from_internal(), y = s.y.from_internal();
        if (fmt == PORLA_POINT_BE64) {
            host::limbs_to_be32(x.v, out + 64 * i);
            host::limbs_to_be32(y.v, out + 64 * i + 32);
        } else {
            memcpy(out + 64 * i, x.v, 32);
            memcpy(out + 64 * i + 32, y.v, 32);
        }
    }
}

}  // namespace

namespace {
// ---------------------------------------------------------------------------- IPA prover support (SURVEY 8(f)3)
// Arithmetic modulo the secp256k1 group order n = 2^256 - C (C has 129 bits): 4 x 64 limbs, products folded with
// hi * C + lo as libsecp256k1's scalar_4x64 does.  Only the prover's scalar bookkeeping runs here (a few hundred
// products per proof, NTL ZZ arithmetic in the reference: Server.hpp:2326-2334, 2344, 2435-2440).
struct Sn {
    uint64_t v[4];
};
const uint64_t kSnN[4] = {0xBFD25E8CD0364141ull, 0xBAAEDCE6AF48A03Bull, 0xFFFFFFFFFFFFFFFEull, 0xFFFFFFFFFFFFFFFFull};
const uint64_t kSnC[3] = {0x402DA1732FC9BEBFull, 0x4551231950B75FC4ull, 0x1ull};

bool sn_geq_n(const uint64_t* a) {
    for (int i = 3; i >= 0; i--)
        if (a[i] != kSnN[i]) return a[i] > kSnN[i];
    return true;
}
void sn_sub_n(uint64_t* a) {
    u128 borrow = 0;
    for (int i = 0; i < 4; i++) {
        u128 d = (u128)a[i] - kSnN[i] - (uint64_t)borrow;
        a[i] = (uint64_t)d;
        borrow = (d >> 64) & 1;
    }
}
// t (len limbs, len <= 8) -> t mod n
Sn sn_reduce(const uint64_t* t, int len) {
    uint64_t cur[9] = {0};
    for (int i = 0; i < len; i++) cur[i] = t[i];
    int n = len;
    while (n > 4) {   // cur = lo + hi * C
        uint64_t nxt[9] = {0};
        for (int i = 0; i < 4; i++) nxt[i] = cur[i];
        const int hl = n - 4;
        for (int i = 0; i < hl; i++) {
            u128 carry = 0;
            for (int j = 0; j < 3; j++) {
                u128 p = (u128)cur[4 + i] * kSnC[j] + nxt[i + j] + (uint64_t)carry;
                nxt[i + j] = (uint64_t)p;
                carry = p >> 64;
            }
            for (int k = i + 3; carry && k < 9; k++) {
                u128 p = (u128)nxt[k] + (uint64_t)carry;
                nxt[k] = (uint64_t)p;
                carry = p >> 64;
            }
        }
        n = 9;
        while (n > 4 && nxt[n - 1] == 0) n--;
        for (int i = 0; i < 9; i++) cur[i] = nxt[i];
    }
    Sn r;
    for (int i = 0; i < 4; i++) r.v[i] = cur[i];
    while (sn_geq_n(r.v)) sn_sub_n(r.v);
    return r;
}
Sn sn_mul(const Sn& a, const Sn& b) {
    uint64_t t[8] = {0};
    for (int i = 0; i < 4; i++) {
        u128 carry = 0;
        for (int j = 0; j < 4; j++) {
            u128 p = (u128)a.v[i] * b.v[j] + t[i + j] + (uint64_t)carry;
            t[i + j] = (uint64_t)p;
            carry = p >> 64;
        }
        t[i + 4] = (uint64_t)carry;
    }
    return sn_reduce(t, 8);
}
Sn sn_add(const Sn& a, const Sn& b) {
    uint64_t t[5];
    u128 carry = 0;
    for (int i = 0; i < 4; i++) {
        u128 p = (u128)a.v[i] + b.v[i] + (uint64_t)carry;
        t[i] = (uint64_t)p;
        carry = p >> 64;
    }
    t[4] = (uint64_t)carry;
    return sn_reduce(t, 5);
}
Sn sn_from_le32(const unsigned char* b) {   // any 256-bit value, reduced
    uint64_t t[4];
    memcpy(t, b, 32);
    return sn_reduce(t, 4);
}
Sn sn_one() { return Sn{{1, 0, 0, 0}}; }
Sn sn_inverse(const Sn& a) {   // a^(n-2)
    uint64_t e[4] = {kSnN[0] - 2, kSnN[1], kSnN[2], kSnN[3]};
    Sn r = sn_one();
    for (int i = 255; i >= 0; i--) {
        r = sn_mul(r, r);
        if ((e[i >> 6] >> (i & 63)) & 1) r = sn_mul(r, a);
    }
    return r;
}

// The reference's Fiat-Shamir object: ONE secp256k1_sha256 written to and finalized repeatedly without
// re-initialisation (Server.hpp:2306-2310, 2386-2387, 2429-2430); finalize wipes the state words and keeps the byte
// counter (hash_impl.h:151-165), which this class reproduces.
struct TranscriptSha256 {
    uint32_t s[8];
    unsigned char buf[64];
    uint64_t bytes = 0;
    TranscriptSha256() {
        static const uint32_t iv[8] = {0x6a09e667u, 0xbb67ae85u, 0x3c6ef372u, 0xa54ff53au, 0x510e527fu, 0x9b05688cu, 0x1f83d9abu, 0x5be0cd19u};
        memcpy(s, iv, sizeof(s));
    }
    static uint32_t rotr(uint32_t x, int n) { return (x >> n) | (x << (32 - n)); }
    void transform(const unsigned char* blk) {
        static const uint32_t K[64] = {
            0x428a2f98u, 0x71374491u, 0xb5c0fbcfu, 0xe9b5dba5u, 0x3956c25bu, 0x59f111f1u, 0x923f82a4u, 0xab1c5ed5u, 0xd807aa98u, 0x12835b01u, 0x243185beu,
            0x550c7dc3u, 0x72be5d74u, 0x80deb1feu, 0x9bdc06a7u, 0xc19bf174u, 0xe49b69c1u, 0xefbe4786u, 0x0fc19dc6u, 0x240ca1ccu, 0x2de92c6fu, 0x4a7484aau,
            0x5cb0a9dcu, 0x76f988dau, 0x983e5152u, 0xa831c66du, 0xb00327c8u, 0xbf597fc7u, 0xc6e00bf3u, 0xd5a79147u, 0x06ca6351u, 0x14292967u, 0x27b70a85u,
            0x2e1b2138u, 0x4d2c6dfcu, 0x53380d13u, 0x650a7354u, 0x766a0abbu, 0x81c2c92eu, 0x92722c85u, 0xa2bfe8a1u, 0xa81a664bu, 0xc24b8b70u, 0xc76c51a3u,
            0xd192e819u, 0xd6990624u, 0xf40e3585u, 0x106aa070u, 0x19a4c116u, 0x1e376c08u, 0x2748774cu, 0x34b0bcb5u, 0x391c0cb3u, 0x4ed8aa4au, 0x5b9cca4fu,
            0x682e6ff3u, 0x748f82eeu, 0x78a5636fu, 0x84c87814u, 0x8cc70208u, 0x90befffau, 0xa4506cebu, 0xbef9a3f7u, 0xc67178f2u};
        uint32_t w[64];
        for (int i = 0; i < 16; i++)
            w[i] = ((uint32_t)blk[4 * i] << 24) | ((uint32_t)blk[4 * i + 1] << 16) | ((uint32_t)blk[4 * i + 2] << 8) | blk[4 * i + 3];
        for (int i = 16; i < 64; i++) {
            uint32_t s0 = rotr(w[i - 15], 7) ^ rotr(w[i - 15], 18) ^ (w[i - 15] >> 3);
            uint32_t s1 = rotr(w[i - 2], 17) ^ rotr(w[i - 2], 19) ^ (w[i - 2] >> 10);
            w[i] = w[i - 16] + s0 + w[i - 7] + s1;
        }
        uint32_t a = s[0], b = s[1], c = s[2], d = s[3], e = s[4], f = s[5], g = s[6], h = s[7];
        for (int i = 0; i < 64; i++) {
            uint32_t t1 = h + (rotr(e, 6) ^ rotr(e, 11) ^ rotr(e, 25)) + ((e & f) ^ (~e & g)) + K[i] + w[i];
            uint32_t t2 = (rotr(a, 2) ^ rotr(a, 13) ^ rotr(a, 22)) + ((a & b) ^ (a & c) ^ (b & c));
            h = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
        }
        s[0] += a; s[1] += b; s[2] += c; s[3] += d; s[4] += e; s[5] += f; s[6] += g; s[7] += h;
    }
    void write(const unsigned char* data, size_t len) {
        size_t fill = (size_t)(bytes & 63);
        bytes += len;
        while (len >= 64 - fill) {
            memcpy(buf + fill, data, 64 - fill);
            data += 64 - fill;
            len -= 64 - fill;
            transform(buf);
            fill = 0;
        }
        if (len) memcpy(buf + fill, data, len);
    }
    void finalize(unsigned char out[32]) {
        unsigned char pad[64] = {0x80};
        unsigned char size[8];
        const uint64_t bits = bytes << 3;
        for (int i = 0; i < 8; i++) size[i] = (unsigned char)(bits >> (8 * (7 - i)));
        write(pad, 1 + ((119 - (size_t)(bytes % 64)) % 64));
        write(size, 8);
        for (int i = 0; i < 8; i++) {
            out[4 * i] = (unsigned char)(s[i] >> 24);
            out[4 * i + 1] = (unsigned char)(s[i] >> 16);
            out[4 * i + 2] = (unsigned char)(s[i] >> 8);
            out[4 * i + 3] = (unsigned char)s[i];
            s[i] = 0;
        }
    }
};

// ---------------------------------------------------------------------------- FFT in the exponent on IPA-mode MACs
// k * p on the host for small stages: k = k1 + k2 lambda (glv_split_secp256k1, the device routine), then joint 2 + 2-bit
// windows over (k1, k2) -- 15 combinations i (+-p) + j (+-phi(p)), 64 steps of two doublings and at most one addition,
// as g1_mul does for BN254.
XYZZ<SF> secp_mul_host(const Affine<SF>& p, const porla_secp256k1_scalar& w) {
    const Sn kn = sn_from_le32((const unsigned char*)w.d);
    if (p.is_inf() || !(kn.v[0] | kn.v[1] | kn.v[2] | kn.v[3])) return XYZZ<SF>::inf();
    uint32_t k[8], k1[4], k2[4], n1, n2;
    memcpy(k, kn.v, 32);
    glv_split_secp256k1(k, k1, k2, n1, n2);
    Affine<SF> p1 = p, p2 = p;
    for (int i = 0; i < 4; i++)
        p2.x.v[i] = (uint64_t)Secp256k1::glv_beta_mont(2 * i) | ((uint64_t)Secp256k1::glv_beta_mont(2 * i + 1) << 32);
    p2.x = p.x * p2.x;
    if (n1) p1.y = p1.y.neg();
    if (n2) p2.y = p2.y.neg();
    XYZZ<SF> tab[16];   // tab[4 j + i] = i p1 + j p2
    tab[0] = XYZZ<SF>::inf();
    for (int i = 1; i < 4; i++) {
        tab[i] = tab[i - 1];
        tab[i].madd(p1);
    }
    for (int j = 1; j < 4; j++)
        for (int i = 0; i < 4; i++) {
            tab[4 * j + i] = tab[4 * (j - 1) + i];
            tab[4 * j + i].madd(p2);
        }
    auto digit = [&](int d) { return ((k1[d >> 4] >> (2 * (d & 15))) & 3u) | (((k2[d >> 4] >> (2 * (d & 15))) & 3u) << 2); };
    int top = 63;
    while (top > 0 && digit(top) == 0) top--;
    XYZZ<SF> r = tab[digit(top)];
    for (int d = top - 1; d >= 0; d--) {
        r = r.dbl().dbl();
        const uint32_t e = digit(d);
        if (e) r.add(tab[e]);
    }
    return r;
}

void gej_from_affine(const Affine<SF>& a, porla_secp256k1_gej* r) {
    uint8_t b[64];
    memcpy(b, a.x.v, 32);
    memcpy(b + 32, a.y.v, 32);
    gej_from_le64(b, r);
}

void butterfly_stage_host(porla_secp256k1_gej* pts, size_t n, size_t m, const porla_secp256k1_scalar* tw) {
    const size_t m2 = m / 2;
    for_each_butterfly_host((int64_t)(n / 2), [&](int64_t lo, int64_t hi) {
        for (int64_t b = lo; b < hi; b++) {
            const size_t j = (size_t)b % m2, k = ((size_t)b / m2) * m + j;
            const Affine<SF> a0 = gej_to_affine(pts + k);
            const XYZZ<SF> t = secp_mul_host(gej_to_affine(pts + k + m2), tw[j]);
            XYZZ<SF> r0 = XYZZ<SF>::from_affine(a0), r1 = r0;
            r0.add(t);
            r1.add(t.neg());
            gej_from_affine(r0.to_affine(), pts + k);
            gej_from_affine(r1.to_affine(), pts + k + m2);
        }
    });
}

// gej as stored -> what k_import_jacobian reads: canonical X, Y, Z (8 LE 32-bit limbs each, zero for infinity) and the
// infinity flags.  The limbs are normalised here; the Jacobian -> affine conversion happens on the device.
void gej_to_device_form(const porla_secp256k1_gej* pts, size_t n, std::vector<uint32_t>* xyz, std::vector<uint8_t>* inf) {
    xyz->assign(24 * n, 0);
    inf->resize(n);
    for (size_t i = 0; i < n; i++) {
        (*inf)[i] = pts[i].infinity ? 1 : 0;
        if ((*inf)[i]) continue;
        fe_to_canonical(&pts[i].x, &(*xyz)[24 * i]);
        fe_to_canonical(&pts[i].y, &(*xyz)[24 * i + 8]);
        fe_to_canonical(&pts[i].z, &(*xyz)[24 * i + 16]);
    }
}

// The same stage on the device: limbs normalised here, Jacobian -> affine in k_import_jacobian, the butterfly kernels of
// butterfly_stage_device, canonical affine back.
void butterfly_stage_gpu(porla_secp256k1_gej* pts, size_t n, size_t m, const porla_secp256k1_scalar* tw) {
    std::vector<uint32_t> xyz;
    std::vector<uint8_t> inf;
    gej_to_device_form(pts, n, &xyz, &inf);
    device_init();
    StagedCall call;
    call.add(96 * n);
    const size_t o_inf = call.add(n), o_tw = call.add(32 * (m / 2)), o_pts = call.add(64 * n), o_flags = call.add(n),
                 o_out = call.add(64 * n);
    uint8_t* d = call.dev();
    cudaStream_t st = call.stream();
    h2d_copy(d, xyz.data(), 96 * n, st);
    PORLA_CUDA(cudaMemcpyAsync(d + o_inf, inf.data(), n, cudaMemcpyHostToDevice, st));
    PORLA_CUDA(cudaMemcpyAsync(d + o_tw, tw, 32 * (m / 2), cudaMemcpyHostToDevice, st));
    PointTable t;
    table_import_jacobian_secp256k1(reinterpret_cast<const uint32_t*>(d), d + o_inf, (uint32_t)n, d + o_pts, d + o_flags, &t, st);
    butterfly_stage_device(&t, (uint32_t)m, d + o_tw, 0, st);
    export_points_device(kCurveSecp256k1, t.d_points, (uint32_t)n, PORLA_POINT_LE64, d + o_out, st);
    std::vector<uint8_t> out(64 * n);
    PORLA_CUDA(cudaMemcpyAsync(out.data(), d + o_out, 64 * n, cudaMemcpyDeviceToHost, st));
    PORLA_CUDA(cudaStreamSynchronize(st));
    gej_batch_from_le64(out.data(), n, pts);
}

// A resident secp256k1 table holding at least n_chunks generators; a staged call indexes terms with 32 bits
bool align_shape_ok(const porla_table* gens, size_t n_chunks, size_t batch) {
    return gens && gens->t.curve == kCurveSecp256k1 && n_chunks && n_chunks <= gens->t.n &&
           (uint64_t)n_chunks * batch < (1ull << 31);
}
}  // namespace

extern "C" {

int porla_secp256k1_butterfly_stage(porla_secp256k1_gej* points, size_t n, size_t m, const porla_secp256k1_scalar* twiddles) {
    if (m < 2 || (m & (m - 1)) || n % m || n > 0xffffffffu) return 0;
    if (n == 0) return 1;
    if ((int64_t)(n / 2) <= host_butterfly_limit(kCurveSecp256k1)) butterfly_stage_host(points, n, m, twiddles);
    else butterfly_stage_gpu(points, n, m, twiddles);
    return 1;
}

int porla_secp256k1_ecmult_multi_var(const porla_secp256k1_callback* error_callback, void* scratch,
                                     porla_secp256k1_gej* r, const porla_secp256k1_scalar* inp_g_sc,
                                     porla_secp256k1_ecmult_multi_callback cb, void* cbdata, size_t n) {
    (void)error_callback;
    (void)scratch;
    gej_set_infinity(r);  // ecmult_impl.h:821
    if (inp_g_sc == NULL && n == 0) return 1;
    std::vector<uint8_t> scalars, points;
    scalars.reserve((n + 1) * 32);
    points.reserve((n + 1) * 64);
    if (inp_g_sc) {
        const uint64_t* d = inp_g_sc->d;
        if (d[0] | d[1] | d[2] | d[3]) {
            scalars.insert(scalars.end(), (const uint8_t*)d, (const uint8_t*)d + 32);
            points.insert(points.end(), kGenLE, kGenLE + 64);
        }
    }
    for (size_t i = 0; i < n; i++) {
        porla_secp256k1_scalar sc;
        porla_secp256k1_ge pt;
        if (!cb(&sc, &pt, i, cbdata)) return 0;  // ecmult_impl.h:696
        if (pt.infinity) continue;               // ecmult_impl.h:500-502 skips them
        if (!(sc.d[0] | sc.d[1] | sc.d[2] | sc.d[3])) continue;
        uint32_t xy[16];
        fe_to_canonical(&pt.x, xy);
        fe_to_canonical(&pt.y, xy + 8);
        scalars.insert(scalars.end(), (const uint8_t*)sc.d, (const uint8_t*)sc.d + 32);
        points.insert(points.end(), (const uint8_t*)xy, (const uint8_t*)xy + 64);
    }
    size_t m = scalars.size() / 32;
    if (m == 0) return 1;
    uint8_t res[64];
    porla_msm_host(PORLA_CURVE_SECP256K1, scalars.data(), points.data(), (int64_t)m, 1, PORLA_SCALAR_LE32,
                   PORLA_POINT_LE64, res);
    gej_from_le64(res, r);
    return 1;
}

// ---- generators resident in HBM (BASELINE north star: "SRS and generator tables resident in HBM, uploaded
// once at init").  Porla's IPA mode multiplies the SAME generator array in every commitment, align_MAC and
// inner-product round (data.pt = &generators[start_chunk]: Server.hpp:347,507,2345,2395, Client.hpp:393,1588);
// the callback adapter above re-uploads them on every call.
porla_table* porla_secp256k1_table_create(const porla_secp256k1_ge* points, size_t n) {
    std::vector<uint8_t> le(n * 64 + 64, 0);
    for (size_t i = 0; i < n; i++) {
        if (points[i].infinity) continue;           // stays 64 zero bytes = infinity
        uint32_t xy[16];
        fe_to_canonical(&points[i].x, xy);
        fe_to_canonical(&points[i].y, xy + 8);
        memcpy(le.data() + 64 * i, xy, 64);
    }
    porla_table* t = porla_table_create(PORLA_CURVE_SECP256K1, le.data(), (int64_t)n, PORLA_POINT_LE64, 0, nullptr);
    // generators are fixed bases: expand them once (small sets such as Porla's 128 get the full look-up table of
    // window multiples, so every commitment / IPA round over them is a plain sum of table entries)
    if (n) porla_table_precompute(t, 0, (int64_t)n, 1, nullptr);
    return t;
}

int porla_secp256k1_ecmult_multi_table_batch(const porla_table* t, size_t first, const porla_secp256k1_scalar* scalars,
                                             size_t n, size_t batch, porla_secp256k1_gej* r) {
    if (!t || t->t.curve != kCurveSecp256k1 || first > t->t.n || n > t->t.n - first) return 0;
    if (batch && n > ((1ull << 31) - 1) / batch) return 0;   // n * batch >= 2^31: a staged call indexes terms with 32 bits
    if (batch == 0) return 1;
    if (n == 0) {
        for (size_t b = 0; b < batch; b++) gej_set_infinity(r + b);
        return 1;
    }
    std::vector<uint8_t> res(64 * batch);
    porla_msm_table_host_scalars_batch(t, (int64_t)first, scalars, (int64_t)n, (int64_t)batch, PORLA_SCALAR_LE32,
                                       PORLA_POINT_LE64, res.data());
    gej_batch_from_le64(res.data(), batch, r);
    return 1;
}

int porla_secp256k1_ecmult_multi_table(const porla_table* t, size_t first, const porla_secp256k1_scalar* scalars, size_t n,
                                       porla_secp256k1_gej* r) {
    gej_set_infinity(r);
    if (n == 0) return 1;
    return porla_secp256k1_ecmult_multi_table_batch(t, first, scalars, n, 1, r);
}

// The client's MAC complements (SURVEY §2 row 10): secp256k1_ecmult_const of one fixed base h by each PRF value, through
// the fixed-base kernel of the KZG twin compute_digest_complement_batch.  porla_secp256k1_table_create(&h, 1) already
// carries what that kernel reads: table_precompute gives a length-1 table the c = 8 look-up table of window multiples.
int porla_secp256k1_ecmult_const_batch(const porla_table* base, const porla_secp256k1_scalar* scalars, size_t n,
                                       porla_secp256k1_gej* r) {
    if (!base || base->t.curve != kCurveSecp256k1 || base->t.n != 1 || n >= (1ull << 31)) return 0;
    if (n == 0) return 1;
    device_init();
    StagedCall call(1, (int64_t)n);
    gej_batch_from_le64(fixed_base_mul_core(call, base, scalars, (int64_t)n, PORLA_SCALAR_LE32, PORLA_POINT_LE64), n, r);
    return 1;
}

// ---- the data side of an IPA-mode server (SURVEY 8(f)2 and (f)4): align_MAC and the audit's aggregation over the resident
// generators, on the kernels and staging of their KZG twins (align_mac_core, audit_aggregate_core), with secp256k1's n as
// GROUP_ORDER (utils.h:32).
int porla_secp256k1_align_mac_batch(const porla_table* gens, size_t n_chunks, void* data, size_t batch,
                                    porla_secp256k1_gej* align_out) {
    if (!align_shape_ok(gens, n_chunks, batch)) return 0;
    if (batch == 0) return 1;
    std::vector<uint8_t> res(64 * batch);
    align_mac_core(kCurveSecp256k1, table_window(gens->t, 0, (int64_t)n_chunks), data, (int64_t)n_chunks, (int64_t)batch,
                   PORLA_POINT_LE64, res.data());
    gej_batch_from_le64(res.data(), batch, align_out);
    return 1;
}

int porla_secp256k1_audit_aggregate(const porla_table* gens, size_t n_chunks, const uint32_t* coefs, const void* blocks,
                                    size_t n, unsigned char* b_out_le32, porla_secp256k1_gej* align_out) {
    if (!align_shape_ok(gens, n_chunks, 1) || n >= (1u << 24)) return 0;
    if (n == 0) {   // B = 0: already reduced, nothing to align
        memset(b_out_le32, 0, 32 * n_chunks);
        gej_set_infinity(align_out);
        return 1;
    }
    std::vector<uint8_t> b_be(32 * n_chunks);
    uint8_t res[64];
    audit_aggregate_core(kCurveSecp256k1, table_window(gens->t, 0, (int64_t)n_chunks), coefs, blocks, (int64_t)n,
                         (int64_t)n_chunks, PORLA_POINT_LE64, b_be.data(), res);
    for (size_t j = 0; j < n_chunks; j++)   // convert_ZZ_to_arr's order: least significant byte first
        for (int k = 0; k < 32; k++) b_out_le32[32 * j + k] = b_be[32 * j + 31 - k];
    gej_from_le64(res, align_out);
    return 1;
}

// The audit's combined_MAC / combined_align and Client::audit on the MACs as stored: the drop-in above needs
// secp256k1_ge, i.e. one host inversion per MAC first (SURVEY App. E); here the Jacobian points go to the device as they
// are (the butterfly stage's route: limbs normalised here, one device inversion per point with z != 1).
int porla_secp256k1_ecmult_multi_gej(const porla_secp256k1_gej* points, const porla_secp256k1_scalar* scalars, size_t n,
                                     size_t nbatch, porla_secp256k1_gej* r) {
    if (nbatch && n >= (1ull << 31) / nbatch) return 0;
    if (n == 0) {
        for (size_t b = 0; b < nbatch; b++) gej_set_infinity(r + b);
        return 1;
    }
    if (nbatch == 0) return 1;
    std::vector<uint32_t> xyz;
    std::vector<uint8_t> inf;
    gej_to_device_form(points, n * nbatch, &xyz, &inf);
    std::vector<uint8_t> res(64 * nbatch);
    msm_host_jacobian_secp256k1(xyz.data(), inf.data(), scalars, (int64_t)n, (int64_t)nbatch, res.data());
    gej_batch_from_le64(res.data(), nbatch, r);
    return 1;
}

size_t porla_secp256k1_inner_product_prove(const porla_table* gens_and_u, size_t n, const unsigned char* a_le32,
                                           const unsigned char* b_le32, unsigned char* proof) {
    // Server::inner_product_prove (Server.hpp:2279-2443) with the generators resident: every L and R is ONE call over
    // the whole table, table entry n holds u and carries the cross term c_L / c_R (the reference adds u^c with
    // secp256k1_ecmult_const, :2376-2378), generators outside the round's blocks carry a zero scalar.
    if (n < 4 || (n & (n - 1)) || (int64_t)(n + 1) != porla_table_len(gens_and_u)) return 0;
    std::vector<Sn> a(n), b(n), xv(n, sn_one());
    for (size_t i = 0; i < n; i++) {
        a[i] = sn_from_le32(a_le32 + 32 * i);
        b[i] = sn_from_le32(b_le32 + 32 * i);
    }
    unsigned char* out = proof;
    Sn ip{{0, 0, 0, 0}};
    for (size_t i = 0; i < n; i++) ip = sn_add(ip, sn_mul(a[i], b[i]));
    memcpy(out, ip.v, 32);   // convert_ZZ_to_arr: eight 32-bit words, least significant first (utils.h:353-364)
    out += 32;
    static const char seed[] = "hash of P, c, etc. all that jazz";
    unsigned char random_str[32];
    TranscriptSha256 sha;
    sha.write((const unsigned char*)seed, 32);
    sha.write(proof, 32);
    sha.finalize(random_str);
    std::vector<Sn> sc(2 * (n + 1));
    size_t k = 1;
    for (size_t half = n / 2; half > 1; half >>= 1, k <<= 1) {
        const Sn x = sn_from_le32(random_str);   // convert_arr_to_ZZ_p (utils.h:384-393), reduced mod n
        const Sn inv_x = sn_inverse(x);
        Sn cL{{0, 0, 0, 0}}, cR{{0, 0, 0, 0}};
        for (size_t i = 0; i < half; i++) {
            cL = sn_add(cL, sn_mul(a[i], b[half + i]));
            cR = sn_add(cR, sn_mul(a[half + i], b[i]));
        }
        // L (odd blocks, a[q], x) and R (even blocks, a[half + q], 1/x) depend on the same challenge: both
        // multi-exponentiations go out as ONE batch of two; their serialisations then enter the transcript in order
        for (int side = 0; side < 2; side++) {
            Sn* v = sc.data() + (size_t)side * (n + 1);
            for (size_t j = 0; j <= n; j++) v[j] = Sn{{0, 0, 0, 0}};
            for (size_t i = 0; i < k; i++) {
                const size_t pos = 2 * i + (side == 0 ? 1 : 0);
                for (size_t j = pos * half, q = 0; j < (pos + 1) * half; j++, q++) {
                    v[j] = sn_mul(a[(side == 0 ? 0 : half) + q], xv[j]);
                    xv[j] = sn_mul(xv[j], side == 0 ? x : inv_x);
                }
            }
            v[n] = side == 0 ? cL : cR;
        }
        uint8_t res[128];
        porla_msm_table_host_scalars_batch(gens_and_u, 0, sc.data(), (int64_t)(n + 1), 2, PORLA_SCALAR_LE32, PORLA_POINT_LE64, res);
        for (int side = 0; side < 2; side++) {
            uint32_t xy[16];
            memcpy(xy, res + 64 * side, 64);
            bool inf = true;
            for (int i = 0; i < 16; i++) inf = inf && xy[i] == 0;
            size_t size = 0;
            if (!inf) {   // secp256k1_eckey_pubkey_serialize, compressed (eckey_impl.h:36-52); infinity serialises to nothing
                out[0] = (xy[8] & 1u) ? 0x03 : 0x02;
                host::limbs_to_be32(xy, out + 1);
                size = 33;
            }
            sha.write(out, size);
            sha.finalize(random_str);
            out += size;
        }
        for (size_t i = 0; i < half; i++) {
            const Sn na = sn_add(sn_mul(a[i], x), sn_mul(a[i + half], inv_x));
            const Sn nb = sn_add(sn_mul(b[i], inv_x), sn_mul(b[i + half], x));
            a[i] = na;
            b[i] = nb;
        }
    }
    for (int i = 0; i < 2; i++) {
        memcpy(out, a[i].v, 32);
        memcpy(out + 32, b[i].v, 32);
        out += 64;
    }
    return (size_t)(out - proof);
}

int porla_secp256k1_inner_product_verify(const porla_table* gens_and_u, size_t n, const porla_secp256k1_gej* commitment,
                                         const unsigned char* proof) {
    // Client::inner_product_verify (Client.hpp:1465-1630).  The reference compares
    //     commitment + c u + sum_rounds (x^2 L + x^-2 R)   with   (a0 b0 + a1 b1) u + sum_even a0 xv_j g_j + sum_odd a1 xv_j g_j ;
    // here the c u term moves to the right, so the left side is the commitment plus ONE variable-base multi-exponentiation
    // over the proof's points and the right side ONE look-up-table multi-exponentiation over the resident table.
    if (n < 4 || (n & (n - 1)) || (int64_t)(n + 1) != porla_table_len(gens_and_u)) return 0;
    size_t rounds = 0;
    for (size_t h = n / 2; h > 1; h >>= 1) rounds++;
    const unsigned char* p = proof;
    const Sn c = sn_from_le32(p);
    p += 32;
    unsigned char random_str[32];
    static const char seed[] = "hash of P, c, etc. all that jazz";
    TranscriptSha256 sha;
    sha.write((const unsigned char*)seed, 32);
    sha.write(proof, 32);
    sha.finalize(random_str);
    std::vector<Sn> xv(n, sn_one()), lr_sc(2 * rounds);
    std::vector<uint8_t> lr_pts(2 * rounds * 64);
    size_t k = 1, r = 0;
    for (size_t half = n / 2; half > 1; half >>= 1, k <<= 1, r++) {
        const Sn x = sn_from_le32(random_str), inv_x = sn_inverse(x);
        for (size_t i = 0; i < k; i++) {
            for (size_t j = (2 * i + 1) * half; j < (2 * i + 2) * half; j++) xv[j] = sn_mul(xv[j], x);
            for (size_t j = 2 * i * half; j < (2 * i + 1) * half; j++) xv[j] = sn_mul(xv[j], inv_x);
        }
        lr_sc[2 * r] = sn_mul(x, x);
        lr_sc[2 * r + 1] = sn_mul(inv_x, inv_x);
        for (int side = 0; side < 2; side++) {   // secp256k1_eckey_pubkey_parse of a compressed point (eckey_impl.h:17-34)
            if (p[0] != 0x02 && p[0] != 0x03) return 0;
            uint32_t xl[8];
            host::be32_to_limbs(p + 1, xl);
            uint32_t pm[8], tmp[8];
            for (int i = 0; i < 8; i++) pm[i] = Secp256k1FpParams::mod(i);
            if (!sub256(tmp, xl, pm)) return 0;                      // x >= p: not a field element
            SF x_;
            memcpy(x_.v, xl, 32);
            SF seven = SF::zero();
            seven.v[0] = 7;
            const SF rhs = x_.sqr() * x_ + seven;
            // y = rhs^((p+1)/4), (p+1)/4 = 2^254 - 2^30 - 244
            static const uint64_t e[4] = {0xffffffffbfffff0cull, 0xffffffffffffffffull, 0xffffffffffffffffull, 0x3fffffffffffffffull};
            SF y = SF::one();
            for (int i = 253; i >= 0; i--) {
                y = y.sqr();
                if ((e[i >> 6] >> (i & 63)) & 1) y = y * rhs;
            }
            if (y.sqr() != rhs) return 0;                            // x is not on the curve
            if ((y.v[0] & 1) != (uint64_t)(p[0] & 1)) y = y.neg();
            memcpy(lr_pts.data() + 64 * (2 * r + side), x_.v, 32);
            memcpy(lr_pts.data() + 64 * (2 * r + side) + 32, y.v, 32);
            sha.write(p, 33);
            sha.finalize(random_str);
            p += 33;
        }
    }
    Sn ab[4];
    for (int i = 0; i < 4; i++) ab[i] = sn_from_le32(p + 32 * i);    // a0 b0 a1 b1
    // right side over the table: a0 xv_j on even generators, a1 xv_j on odd ones, (a0 b0 + a1 b1 - c) on u
    std::vector<Sn> sc(n + 1);
    for (size_t j = 0; j < n; j++) sc[j] = sn_mul(ab[(j & 1) ? 2 : 0], xv[j]);
    Sn neg_c{{0, 0, 0, 0}};
    if (c.v[0] | c.v[1] | c.v[2] | c.v[3]) {
        u128 borrow = 0;
        for (int i = 0; i < 4; i++) {
            u128 d = (u128)kSnN[i] - c.v[i] - (uint64_t)borrow;
            neg_c.v[i] = (uint64_t)d;
            borrow = (d >> 64) & 1;
        }
    }
    sc[n] = sn_add(sn_add(sn_mul(ab[0], ab[1]), sn_mul(ab[2], ab[3])), neg_c);
    uint8_t rhs64[64], lr64[64];
    porla_msm_table_host_scalars(gens_and_u, 0, sc.data(), (int64_t)(n + 1), PORLA_SCALAR_LE32, PORLA_POINT_LE64, rhs64);
    porla_msm_host(PORLA_CURVE_SECP256K1, lr_sc.data(), lr_pts.data(), (int64_t)(2 * rounds), 1, PORLA_SCALAR_LE32, PORLA_POINT_LE64, lr64);
    // left side: commitment (Jacobian, any field magnitude) + the L / R combination, on the host
    auto load_affine = [](const uint8_t* b) {
        Affine<SF> a;
        memcpy(a.x.v, b, 32);
        memcpy(a.y.v, b + 32, 32);
        return a;
    };
    XYZZ<SF> lhs = XYZZ<SF>::from_affine(gej_to_affine(commitment));
    lhs.madd(load_affine(lr64));             // all-zero bytes = infinity: madd ignores it
    const Affine<SF> l = lhs.to_affine(), rr = load_affine(rhs64);
    return l.x == rr.x && l.y == rr.y ? 1 : 0;
}

int porla_secp256k1_gej_serialize(const porla_secp256k1_gej* a, unsigned char out33[33]) {
    if (a->infinity) return 0;
    const Affine<SF> p = gej_to_affine(a);
    uint32_t x[8];
    memcpy(x, p.x.v, 32);
    out33[0] = (p.y.v[0] & 1u) ? 0x03 : 0x02;  // SECP256K1_TAG_PUBKEY_ODD / EVEN
    host::limbs_to_be32(x, out33 + 1);
    return 1;
}

void porla_debug_point_add_host(int curve, const void* a, const void* b, int64_t n, int point_fmt, void* out) {
    if (curve == PORLA_CURVE_BN254) point_add_host<Bn254>((const uint8_t*)a, (const uint8_t*)b, n, point_fmt, (uint8_t*)out);
    else point_add_host<Secp256k1>((const uint8_t*)a, (const uint8_t*)b, n, point_fmt, (uint8_t*)out);
}

}  // extern "C"
