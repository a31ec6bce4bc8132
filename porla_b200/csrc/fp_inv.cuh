// Modular inversion without multiplications on the field's multiplier: binary extended GCD in the style of
// T. Pornin, "Optimized Binary GCD for Modular Inversion" (2020).  It is Fp::inverse on the device, behind every
// conversion to affine coordinates (to_affine, k_fixed_base_mul, the butterfly kernels, k_lut_build).  A Fermat inversion
// (~300 field products) runs on the multiplier pipe (IMAD.WIDE) that bounds those kernels, while this routine is ~23 k
// instructions, mostly plain ALU work (shifts, adds, selects), and overlaps with other warps' field products.  Measured on a
// B200 (tools/inv_probe.py): 77 k cycles on a lone warp against 272 k for the Fermat inversion; 11.7 k SM-cycles per warp
// under load against 42 k.
//
//   a = y, b = m, u = 1, v = 0;   invariants  a = u y,  b = v y  (mod m)
//   repeat: 30 steps of the binary GCD on 64-bit APPROXIMATIONS of (a, b) -- their top 34 bits and their low 30 bits --
//           which only record the update factors  (a, b) <- ((a f0 + b g0) / 2^30, (a f1 + b g1) / 2^30),  |f|, |g| <= 2^30;
//           then apply the factors to the full-size a, b (exact division) and to u, v (division by 2^30 mod m, Montgomery
//           style).  A value that comes out negative is negated together with its co-factor.
//   after ceil(2 bits / 30) + 1 rounds  b = gcd = 1  and  v = y^-1.  Extra rounds are harmless (a = 0 stays 0).
//
// Plain C++ (no inline PTX): the same code is exercised on the host by tests/test_fp_inv_host.py.
// Included by fp.cuh right after the raw 256-bit helpers (it needs sub256 and the modulus parameters only).
#pragma once

namespace porla {

PORLA_HD constexpr uint32_t neg_inv_u32(uint32_t m0) {   // -m0^-1 mod 2^32 for odd m0 (Newton: 3 -> 6 -> 12 -> 24 -> 48 bits)
    uint32_t x = m0;
    x *= 2u - m0 * x;
    x *= 2u - m0 * x;
    x *= 2u - m0 * x;
    x *= 2u - m0 * x;
    return 0u - x;
}

constexpr int kGcdSteps = 30;

// t (10 limbs, two's complement) = a f + b g,  a, b unsigned 8 limbs, f, g signed
PORLA_HD void gcd_lincomb(const uint32_t* a, const uint32_t* b, int32_t f, int32_t g, uint32_t* t) {
    const uint32_t fu = (uint32_t)f, gu = (uint32_t)g;
    uint32_t p[9], q[9];
    uint64_t c1 = 0, c2 = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        c1 += (uint64_t)a[i] * fu;
        p[i] = (uint32_t)c1;
        c1 >>= 32;
        c2 += (uint64_t)b[i] * gu;
        q[i] = (uint32_t)c2;
        c2 >>= 32;
    }
    p[8] = (uint32_t)c1;
    q[8] = (uint32_t)c2;
    uint64_t c = 0;
#pragma unroll
    for (int i = 0; i < 9; i++) {
        c += (uint64_t)p[i] + q[i];
        t[i] = (uint32_t)c;
        c >>= 32;
    }
    t[9] = (uint32_t)c;
    // f, g were multiplied as unsigned: take a * 2^32 (b * 2^32) back where they are negative
    const uint32_t mf = f < 0 ? 0xffffffffu : 0u, mg = g < 0 ? 0xffffffffu : 0u;
    uint64_t br1 = 0, br2 = 0;
#pragma unroll
    for (int i = 1; i < 10; i++) {
        const uint32_t sa = i <= 8 ? (a[i - 1] & mf) : 0u, sb = i <= 8 ? (b[i - 1] & mg) : 0u;
        uint64_t d = (uint64_t)t[i] - sa - br1;
        br1 = (d >> 63) & 1u;
        uint64_t e = (uint64_t)(uint32_t)d - sb - br2;
        br2 = (e >> 63) & 1u;
        t[i] = (uint32_t)e;
    }
}

// r (8 limbs) = |t / 2^30| for a 10-limb two's complement t that is divisible by 2^30 and below 2^286 in magnitude;
// returns 1 when t was negative
PORLA_HD uint32_t gcd_shift_abs(const uint32_t* t, uint32_t* r) {
    const uint32_t neg = t[9] >> 31;
    const uint32_t x = neg ? 0xffffffffu : 0u;
    uint64_t c = neg;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const uint32_t w = (t[i] >> kGcdSteps) | (t[i + 1] << (32 - kGcdSteps));
        c += (uint64_t)(w ^ x);
        r[i] = (uint32_t)c;
        c >>= 32;
    }
    return neg;
}

// out = (u f + v g) / 2^30 mod m  (negated when `negate`);  u, v in [0, m);  mu = m - u, mv = m - v
template <class P>
PORLA_HD void gcd_lincomb_mod(const uint32_t* u, const uint32_t* v, const uint32_t* mu, const uint32_t* mv, int32_t f, int32_t g,
                              uint32_t negate, uint32_t* out) {
    const uint32_t af = (uint32_t)(f < 0 ? -f : f), ag = (uint32_t)(g < 0 ? -g : g);
    uint32_t t[10];
    {
        uint64_t c1 = 0, c2 = 0;
        uint32_t p[9], q[9];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const uint32_t uu = f < 0 ? mu[i] : u[i], vv = g < 0 ? mv[i] : v[i];
            c1 += (uint64_t)uu * af;
            p[i] = (uint32_t)c1;
            c1 >>= 32;
            c2 += (uint64_t)vv * ag;
            q[i] = (uint32_t)c2;
            c2 >>= 32;
        }
        p[8] = (uint32_t)c1;
        q[8] = (uint32_t)c2;
        uint64_t c = 0;
#pragma unroll
        for (int i = 0; i < 9; i++) {
            c += (uint64_t)p[i] + q[i];
            t[i] = (uint32_t)c;
            c >>= 32;
        }
        t[9] = (uint32_t)c;
    }
    // make the low 30 bits vanish: t += ((t * -m^-1) mod 2^30) * m
    constexpr uint32_t ninv = neg_inv_u32(P::mod(0));
    const uint32_t qq = (t[0] * ninv) & ((1u << kGcdSteps) - 1u);
    {
        uint64_t c = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            c += (uint64_t)qq * P::mod(i) + t[i];
            t[i] = (uint32_t)c;
            c >>= 32;
        }
        c += t[8];
        t[8] = (uint32_t)c;
        t[9] += (uint32_t)(c >> 32);
    }
    uint32_t r[9];
#pragma unroll
    for (int i = 0; i < 9; i++) r[i] = (t[i] >> kGcdSteps) | (t[i + 1] << (32 - kGcdSteps));
    // r < 3 m: two conditional subtractions
#pragma unroll
    for (int k = 0; k < 2; k++) {
        uint32_t d[9];
        uint64_t br = 0;
#pragma unroll
        for (int i = 0; i < 9; i++) {
            uint64_t e = (uint64_t)r[i] - (i < 8 ? P::mod(i) : 0u) - br;
            d[i] = (uint32_t)e;
            br = (e >> 63) & 1u;
        }
        if (!br) {
#pragma unroll
            for (int i = 0; i < 9; i++) r[i] = d[i];
        }
    }
    if (negate) {
        uint32_t nz = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) nz |= r[i];
        uint64_t br = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            uint64_t e = (uint64_t)P::mod(i) - r[i] - br;
            out[i] = nz ? (uint32_t)e : 0u;
            br = (e >> 63) & 1u;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 8; i++) out[i] = r[i];
    }
}

// out = x^-1 mod p on plain integers (x in [0, p), 8 LE limbs); 0 -> 0
template <class P, int kBits>
PORLA_HD void fp_inverse_plain(const uint32_t* x, uint32_t* out) {
    constexpr int kRounds = (2 * kBits + kGcdSteps - 1) / kGcdSteps + 1;
    uint32_t a[8], b[8], u[8], v[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        a[i] = x[i];
        b[i] = P::mod(i);
        u[i] = i == 0 ? 1u : 0u;
        v[i] = 0u;
    }
#pragma unroll 1
    for (int round = 0; round < kRounds; round++) {
        // ---- 64-bit approximations: top 34 bits (aligned to the longer of the two) and low 30 bits
        uint32_t ah = a[1], am = a[0], al = 0, bh = b[1], bm = b[0], bl = 0;
        bool found = false;
#pragma unroll
        for (int j = 7; j >= 2; j--) {
            const bool nz = (a[j] | b[j]) != 0u;
            const bool take = nz && !found;
            ah = take ? a[j] : ah;
            am = take ? a[j - 1] : am;
            al = take ? a[j - 2] : al;
            bh = take ? b[j] : bh;
            bm = take ? b[j - 1] : bm;
            bl = take ? b[j - 2] : bl;
            found = found || nz;
        }
        uint32_t xa_hi, xa_lo, xb_hi, xb_lo;
        if (found) {
            const uint32_t top = ah | bh;            // != 0 here
#ifdef __CUDA_ARCH__
            const int s = __clz((int)top);
#else
            const int s = __builtin_clz(top);
#endif
            const uint32_t a_hi = s ? ((ah << s) | (am >> (32 - s))) : ah, a_lo = s ? ((am << s) | (al >> (32 - s))) : am;
            const uint32_t b_hi = s ? ((bh << s) | (bm >> (32 - s))) : bh, b_lo = s ? ((bm << s) | (bl >> (32 - s))) : bm;
            xa_hi = a_hi;
            xa_lo = (a_lo & 0xc0000000u) | (a[0] & 0x3fffffffu);
            xb_hi = b_hi;
            xb_lo = (b_lo & 0xc0000000u) | (b[0] & 0x3fffffffu);
        } else {
            xa_hi = a[1];
            xa_lo = a[0];
            xb_hi = b[1];
            xb_lo = b[0];
        }
        // ---- 30 binary-GCD steps on the approximations
        int32_t f0 = 1, g0 = 0, f1 = 0, g1 = 1;
#pragma unroll 2
        for (int k = 0; k < kGcdSteps; k++) {
            const bool odd = (xa_lo & 1u) != 0u;
            const bool lt = xa_hi < xb_hi || (xa_hi == xb_hi && xa_lo < xb_lo);
            const bool sw = odd && lt;
            const uint32_t ta_hi = sw ? xb_hi : xa_hi, ta_lo = sw ? xb_lo : xa_lo;
            xb_hi = sw ? xa_hi : xb_hi;
            xb_lo = sw ? xa_lo : xb_lo;
            const int32_t tf = sw ? f1 : f0, tg = sw ? g1 : g0;
            f1 = sw ? f0 : f1;
            g1 = sw ? g0 : g1;
            // a -= b, (f0, g0) -= (f1, g1) when a is odd
            const uint32_t sb_lo = odd ? xb_lo : 0u, sb_hi = odd ? xb_hi : 0u;
            const uint32_t d_lo = ta_lo - sb_lo;
            const uint32_t d_hi = ta_hi - sb_hi - (ta_lo < sb_lo ? 1u : 0u);
            f0 = tf - (odd ? f1 : 0);
            g0 = tg - (odd ? g1 : 0);
            xa_lo = (d_lo >> 1) | (d_hi << 31);
            xa_hi = d_hi >> 1;
            f1 += f1;
            g1 += g1;
        }
        // ---- apply to the full-size values
        uint32_t ta[10], tb[10], na[8], nb[8], nu[8], nv[8], mu[8], mv[8], m[8];
        gcd_lincomb(a, b, f0, g0, ta);
        gcd_lincomb(a, b, f1, g1, tb);
        const uint32_t nega = gcd_shift_abs(ta, na), negb = gcd_shift_abs(tb, nb);
#pragma unroll
        for (int i = 0; i < 8; i++) m[i] = P::mod(i);
        sub256(mu, m, u);
        sub256(mv, m, v);
        gcd_lincomb_mod<P>(u, v, mu, mv, f0, g0, nega, nu);
        gcd_lincomb_mod<P>(u, v, mu, mv, f1, g1, negb, nv);
#pragma unroll
        for (int i = 0; i < 8; i++) {
            a[i] = na[i];
            b[i] = nb[i];
            u[i] = nu[i];
            v[i] = nv[i];
        }
    }
#pragma unroll
    for (int i = 0; i < 8; i++) out[i] = v[i];
}

#ifdef __CUDACC__
// one copy per field in device code (the routine is ~3 k instructions)
template <class P>
__device__ __noinline__ void fp_inverse_plain_outlined(const uint32_t* x, uint32_t* out) {
    fp_inverse_plain<P, P::kBits>(x, out);
}
#endif

}  // namespace porla
