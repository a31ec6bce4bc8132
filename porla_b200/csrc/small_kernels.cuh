// Latency-oriented kernels for Porla-shaped calls: a few hundred terms per MSM, one MSM (or a handful)
// per call.  The reference issues them one at a time: the 128..766-term audit aggregation
// (/root/reference/porla/Server/Server.hpp:900-901, Client.hpp:795 -> compute_multi_exp, main.go:119-138)
// and the 128-term commitments over the SRS (Server.hpp:558 -> compute_digest_from_srs, main.go:104-116;
// create_proof, main.go:154-175).  At that size the sort / accumulate / reduce pipeline is a chain of
// ~15 dependent launches; here one launch does the whole MSM as a TREE SUM, whose depth (the only thing
// that matters when every warp has a multiplier pipe to itself) is ~log2(terms) XYZZ additions.
//
//   k_small_bits  variable bases.  Window = one bit: W_b = sum of the points whose scalar has bit b set.
//                 No buckets, no recoding, no bucket reduction; the host's Horner pass (one doubling per
//                 bit) combines the W_b.  Work n * bits / 2 mixed additions, fine for n * bits <= 2^18.
//   k_lut_sum     fixed bases (SRS / generator tables).  A look-up table resident in HBM holds EVERY
//                 multiple d * 2^(c*w) * P_i (1 <= d <= 2^(c-1)); an MSM is the sum of n * nwin table
//                 entries, no doublings at all.  128 bases, c = 8: 32 windows x 128 multiples x 128 bases
//                 x 64 B = 32 MiB (L2-resident on a B200).  Layout [base][window][multiple]: the entries one
//                 scalar touches lie within nwin * 2^(c-1) * 64 B, and a large batch walks the table one slab
//                 of 128 bases at a time (blocks of the same bases are adjacent in the grid), which keeps the
//                 gathers of a 73 GB table (4096 bases, c = 15) inside a 2.3 GB working set.
//   k_lut_build   fills that table from the fixed-base window expansion (k_precompute_windows).
//
// Both sum kernels: a block of 128 threads folds its terms with mixed additions, then a shared-memory
// tree; when an MSM (window) spans several blocks, the last block to arrive (one atomic ticket per
// output) folds the block partials, so a single launch produces the final XYZZ sums.
#pragma once
#include "msm_kernels.cuh"
#include "quad.cuh"

namespace porla {

constexpr int kTreeThreads = 128;

// ONE copy of the XYZZ addition for the trees below (the kernels already inline the mixed addition of their main
// loop; a second and third inlined 14-product addition made the batched look-up sums instruction-fetch bound:
// ncu stall_no_instructions on top, 60 % multiplier-pipe utilisation).
template <class F>
__device__ __noinline__ void xyzz_add_shared(XYZZ<F>* a, const XYZZ<F>* b) {
    XYZZ<F> r = *a;
    r.add(*b);
    *a = r;
}

// Sum of v over the first `count` threads of the block (count <= kTreeThreads); every thread must call.
// The result is returned to thread 0.  Each addition of the tree is carried by FOUR lanes (quad.cuh: 2.35 us against 6.1 us
// for the dependent addition of a lone warp), so a level of up to 32 additions is one round of the block's 32 quads and the
// 7 levels of a 128-value sum take 8 rounds of ~2.4 us instead of 7 additions of ~6.3 us.
template <class F>
PORLA_D XYZZ<F> block_tree_sum(const XYZZ<F>& v, uint32_t count, XYZZ<F>* sh) {
    sh[threadIdx.x] = v;
    __syncthreads();
    uint32_t o = 1;
    while (o < count) o <<= 1;
    const uint32_t quad = threadIdx.x >> 2, role = threadIdx.x & 3;
#pragma unroll 1
    for (o >>= 1; o > 0; o >>= 1) {
#pragma unroll 1
        for (uint32_t base = 0; base < o; base += kTreeThreads / 4) {
            const uint32_t i = base + quad;
            const bool act = i < o && i + o < count;
            if (__any_sync(kFullMask, act)) {                  // warp-uniform: a warp without work skips the round
                QuadPoint<F> a = QuadPoint<F>::inf(), b = QuadPoint<F>::inf();
                if (act) {
                    a.c = reinterpret_cast<const F*>(&sh[i])[role];
                    b.c = reinterpret_cast<const F*>(&sh[i + o])[role];
                }
                a = quad_add_nl(a, b);                         // one outlined copy: the call is short, the code stays in the i-cache
                if (act) reinterpret_cast<F*>(&sh[i])[role] = a.c;
            }
        }
        __syncthreads();
    }
    XYZZ<F> r = sh[0];
    __syncthreads();
    return r;
}

// Cross-block fold: block `blk` of `nblk` contributes `v` (valid in thread 0) to output slot `slot`.
// The last block to take a ticket sums all contributions and stores the result.
template <class F>
PORLA_D void fold_blocks(const XYZZ<F>& v, uint32_t slot, uint32_t blk, uint32_t nblk, XYZZ<F>* __restrict__ partials,
                         uint32_t* __restrict__ tickets, XYZZ<F>* __restrict__ out, XYZZ<F>* sh) {
    if (nblk == 1) {
        if (threadIdx.x == 0) st16(out + slot, v);
        return;
    }
    __shared__ uint32_t s_last;
    if (threadIdx.x == 0) {
        st16(partials + (size_t)slot * nblk + blk, v);
        __threadfence();
        s_last = atomicAdd(tickets + slot, 1u) == nblk - 1 ? 1u : 0u;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    XYZZ<F> acc = XYZZ<F>::inf();
    const volatile uint4* src = reinterpret_cast<const volatile uint4*>(partials + (size_t)slot * nblk);
    for (uint32_t k = threadIdx.x; k < nblk; k += kTreeThreads) {   // volatile: written by other SMs during this launch
        XYZZ<F> p;
        uint4* d = reinterpret_cast<uint4*>(&p);
#pragma unroll
        for (int q = 0; q < 8; q++) {
            d[q].x = src[k * 8 + q].x; d[q].y = src[k * 8 + q].y; d[q].z = src[k * 8 + q].z; d[q].w = src[k * 8 + q].w;
        }
        xyzz_add_shared(&acc, &p);
    }
    XYZZ<F> r = block_tree_sum(acc, nblk < (uint32_t)kTreeThreads ? nblk : (uint32_t)kTreeThreads, sh);
    if (threadIdx.x == 0) st16(out + slot, r);
}

// ---------------------------------------------------------------------------- variable bases, one bit per window
// grid = (chunks of 2*kTreeThreads points, nbits, nbatch); out[m * nbits + b] = W_b of MSM m.
template <class C>
__global__ void __launch_bounds__(kTreeThreads)
k_small_bits(const Affine<typename C::F>* __restrict__ points, const uint8_t* __restrict__ inf_flags,
             const uint8_t* __restrict__ scalars, int big_endian, uint32_t n, int shared_points,
             XYZZ<typename C::F>* __restrict__ partials, uint32_t* __restrict__ tickets,
             XYZZ<typename C::F>* __restrict__ out) {
    using F = typename C::F;
    __shared__ XYZZ<F> sh[kTreeThreads];
    const uint32_t bit = blockIdx.y, m = blockIdx.z, nbits = gridDim.y;
    XYZZ<F> acc = XYZZ<F>::inf();
#pragma unroll 1
    for (int k = 0; k < 2; k++) {
        const uint32_t i = blockIdx.x * (2 * kTreeThreads) + k * kTreeThreads + threadIdx.x;
        if (i >= n) continue;
        const size_t pidx = shared_points ? i : (size_t)m * n + i;
        if (inf_flags && inf_flags[pidx]) continue;
        uint32_t s[8];
        const uint32_t flip = canonical_scalar<C>(scalars, (size_t)m * n + i, big_endian, s);
        if (!((s[bit >> 5] >> (bit & 31)) & 1u)) continue;
        Affine<F> p = ld16(points + pidx);
        if (flip) p.y = p.y.neg();
        acc.madd(p);
    }
    XYZZ<F> r = block_tree_sum(acc, kTreeThreads, sh);
    fold_blocks(r, m * nbits + bit, blockIdx.x, gridDim.x, partials, tickets, out, sh);
}

// ---------------------------------------------------------------------------- fixed bases, full look-up table
// lut[((i * nwin + w) << (c-1)) + d - 1] = d * 2^(c*w) * P_i.
// Signed c-bit digits as in k_digits.  The carry into window w is 1 exactly when the low c*w bits of the
// scalar exceed H_w = sum_{j<w} 2^(c-1) * 2^(c*j) (the value whose every digit sits on the rounding
// boundary), so a thread can start at any window without walking the lower ones.
PORLA_D uint32_t carry_into_window(const uint32_t* s, int c, int w) {
    if (w == 0) return 0;
    const int nb = c * w;                       // compare the low nb bits with H_w, from the top limb down
    for (int limb = 7; limb >= 0; limb--) {
        if (limb * 32 >= nb) continue;
        uint32_t h = 0;
        for (int j = 0; j < w; j++) {
            int pos = c * j + c - 1;
            if ((pos >> 5) == limb) h |= 1u << (pos & 31);
        }
        uint32_t v = s[limb];
        if (nb - limb * 32 < 32) v &= (1u << (nb - limb * 32)) - 1u;
        if (v != h) return v > h ? 1u : 0u;
    }
    return 0;
}

// Signed c-bit digit of window w of a canonical scalar s (9 limbs, s[8] = 0, so the top window may read past bit 255).
// `carry` enters as the carry into window w (carry_into_window, or the previous call's) and leaves as the carry into
// w + 1.  Returns |d_w| in [0, 2^(c-1)]; neg = 1 when d_w < 0.
PORLA_D uint32_t signed_digit(const uint32_t* s, int c, int w, uint32_t& carry, uint32_t& neg) {
    const uint32_t half = 1u << (c - 1), mask = (1u << c) - 1u;
    const uint32_t pos = (uint32_t)w * c, word = pos >> 5, sft = pos & 31;
    const uint32_t lo = s[word < 8 ? word : 8], hi = s[word < 7 ? word + 1 : 8];
    const uint32_t d = (__funnelshift_r(lo, hi, sft) & mask) + carry;
    neg = d > half;
    carry = neg;
    return neg ? ((1u << c) - d) : d;
}

// Thread t of MSM m folds the pairs [t*K, (t+1)*K) of the n*nwin (scalar i, window w) pairs, p = i*nwin + w, whose
// table entry is lut[(p << (c-1)) + |digit| - 1].  Grid: (blocks per MSM, nbatch), or (nbatch, blocks per MSM) when
// m_major (large batches: concurrently resident blocks then read the same slab of bases).  out[m] = the MSM's sum.
// The next entry is fetched before the current mixed addition: the loads depend on the digits only.
template <class C>
__global__ void __launch_bounds__(kTreeThreads)
k_lut_sum(const Affine<typename C::F>* __restrict__ lut, int c, int nwin,
          const uint8_t* __restrict__ scalars, int big_endian, uint32_t n, uint32_t K, int m_major,
          XYZZ<typename C::F>* __restrict__ partials, uint32_t* __restrict__ tickets,
          XYZZ<typename C::F>* __restrict__ out) {
    using F = typename C::F;
    __shared__ XYZZ<F> sh[kTreeThreads];
    const uint32_t m = m_major ? blockIdx.x : blockIdx.y;
    const uint32_t blk = m_major ? blockIdx.y : blockIdx.x;
    const uint32_t nblk = m_major ? gridDim.y : gridDim.x;
    const uint32_t total = n * (uint32_t)nwin;
    uint32_t p = (blk * kTreeThreads + threadIdx.x) * K;
    const uint32_t p_end = p + K < total ? p + K : total;
    XYZZ<F> acc = XYZZ<F>::inf();
    if (p < total) {
        uint32_t i = p / (uint32_t)nwin;
        int w = (int)(p - i * (uint32_t)nwin);
        uint32_t s[9];
        uint32_t flip = canonical_scalar<C>(scalars, (size_t)m * n + i, big_endian, s);
        s[8] = 0;
        uint32_t carry = carry_into_window(s, c, w);
        Affine<F> cur = Affine<F>::inf();     // entry of the previous pair, added one iteration later
#pragma unroll 1
        for (; p <= p_end; p++) {             // one extra turn adds the last entry (a single copy of the mixed addition)
            Affine<F> nxt = Affine<F>::inf();
            if (p < p_end) {
                uint32_t dneg;
                const uint32_t mag = signed_digit(s, c, w, carry, dneg);
                if (mag != 0) {
                    nxt = ld16(lut + (((size_t)p << (c - 1)) + (mag - 1)));
                    if (dneg ^ flip) nxt.y = nxt.y.neg();
                }
                if (++w == nwin) {
                    w = 0;
                    carry = 0;
                    if (++i < n && p + 1 < p_end) {
                        flip = canonical_scalar<C>(scalars, (size_t)m * n + i, big_endian, s);
                        s[8] = 0;
                    }
                }
            }
            acc.madd(cur);
            cur = nxt;
        }
    }
    XYZZ<F> r = block_tree_sum(acc, kTreeThreads, sh);
    fold_blocks(r, m, blk, nblk, partials, tickets, out, sh);
}

// ---------------------------------------------------------------------------- one fixed base, many scalars
// out[i] = k_i * B from the look-up table of ONE base (the table of a length-1 PointTable: lut[(w << (c-1)) + d - 1] =
// d * 2^(c*w) * B).  One thread per scalar: the signed digits of k_lut_sum (same sign flip for secp256k1 scalars above
// n/2), at most nwin mixed additions and no doublings, then the affine normalisation and the caller's output format.
constexpr int kFixedBaseThreads = 128;
template <class C>
__global__ void __launch_bounds__(kFixedBaseThreads)
k_fixed_base_mul(const Affine<typename C::F>* __restrict__ lut, int c, int nwin, const uint8_t* __restrict__ scalars,
                 int big_endian, uint32_t n, int out_fmt, uint8_t* __restrict__ out) {
    using F = typename C::F;
    const uint32_t i = blockIdx.x * kFixedBaseThreads + threadIdx.x;
    if (i >= n) return;
    uint32_t s[9];
    const uint32_t flip = canonical_scalar<C>(scalars, i, big_endian, s);
    s[8] = 0;
    uint32_t carry = 0;
    XYZZ<F> acc = XYZZ<F>::inf();
    Affine<F> cur = Affine<F>::inf();     // entry of the previous window, added one iteration later
#pragma unroll 1
    for (int w = 0; w <= nwin; w++) {     // one extra turn adds the last entry (a single copy of the mixed addition)
        Affine<F> nxt = Affine<F>::inf();
        if (w < nwin) {
            uint32_t neg;
            const uint32_t mag = signed_digit(s, c, w, carry, neg);
            if (mag != 0) {
                nxt = ld16(lut + (((size_t)w << (c - 1)) + (mag - 1)));
                if (neg ^ flip) nxt.y = nxt.y.neg();
            }
        }
        acc.madd(cur);
        cur = nxt;
    }
    // One inversion per thread.  A block-wide batch inversion (Montgomery's trick over the threads' zzz in shared memory)
    // measured no faster at 2^20 and 2^24 scalars and 13 % slower at 2^16 (BN254) on a B200: profiles/r03_fixed_base_mul_inversion.txt.
    const Affine<F> a = acc.to_affine();
    const F x = a.x.from_internal(), y = a.y.from_internal();
    store_u256(out, 2 * (size_t)i, out_fmt == kPointBE64, x.v);
    store_u256(out, 2 * (size_t)i + 1, out_fmt == kPointBE64, y.v);
}

// One thread per (window, base): the 2^(c-1) multiples of Q = 2^(c*w) * P_i, normalised to affine kLutChunk at a
// time with ONE inversion per chunk (Montgomery's trick on the zzz coordinates): ~36 field products per entry, so
// the 1.1 * 10^9 entries of a 4096-base, c = 15 table (73 GB) are a fraction of a second of one-time work.
constexpr int kLutChunk = 16;
template <class C>
__global__ void __launch_bounds__(128)
k_lut_build(const Affine<typename C::FC>* __restrict__ fb_points, const uint8_t* __restrict__ inf_flags, uint32_t n,
            int c, int nwin, Affine<typename C::FC>* __restrict__ lut) {
    using F = typename C::FC;
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * (uint32_t)nwin) return;
    const uint32_t i = t % n;
    const uint32_t count = 1u << (c - 1);
    const uint32_t w = t / n;                          // fb_points is [window][base], the table [base][window][multiple]
    Affine<F>* dst = lut + (((size_t)i * nwin + w) << (c - 1));
    const Affine<F> q = ld16(fb_points + t);
    if (q.is_inf() || (inf_flags && inf_flags[i])) {
        for (uint32_t d = 0; d < count; d++) st16(dst + d, Affine<F>::inf());
        return;
    }
    st16(dst, q);
    XYZZ<F> r = XYZZ<F>::from_affine(q);
    XYZZ<F> buf[kLutChunk];
    F prefix[kLutChunk];
    for (uint32_t d0 = 1; d0 < count; d0 += kLutChunk) {
        const uint32_t m = count - d0 < (uint32_t)kLutChunk ? count - d0 : (uint32_t)kLutChunk;
        F acc = F::one();
        for (uint32_t j = 0; j < m; j++) {
            r.madd(q);                 // (d0 + j + 1) * Q: never infinity below the group order
            buf[j] = r;
            acc = acc * r.zzz;
            prefix[j] = acc;
        }
        F inv = acc.inverse();         // 1 / (zzz_0 ... zzz_{m-1})
        for (uint32_t j = m; j-- > 0;) {
            const F i3 = j ? prefix[j - 1] * inv : inv;     // 1 / zzz_j
            inv = inv * buf[j].zzz;
            const F tt = buf[j].zz * i3;                    // 1 / zz_j = (zz_j / zzz_j)^2
            Affine<F> a;
            a.x = buf[j].x * tt.sqr();
            a.y = buf[j].y * i3;
            st16(dst + d0 + j, a);
        }
    }
}

}  // namespace porla
