// Templated host drivers of the kernels in msm_kernels.cuh; instantiated once per curve in
// msm_bn254.cu / msm_secp.cu so the two curves compile in parallel.
#pragma once
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <type_traits>

#include "arena.h"
#include "msm.h"
#include "msm_kernels.cuh"
#include "small_kernels.cuh"

namespace porla {

extern std::atomic<uint64_t> g_launches;
#define LAUNCHED() (g_launches.fetch_add(1, std::memory_order_relaxed))



template <class C> struct CurveIdOf;
template <> struct CurveIdOf<Bn254> { static constexpr int value = kCurveBn254; };
template <> struct CurveIdOf<Secp256k1> { static constexpr int value = kCurveSecp256k1; };

// ---------------------------------------------------------------------------- tables
template <class C>
void import_into_impl(const uint8_t* d_bytes, int fmt, uint32_t n, void* d_points_out, uint8_t* d_flags_out,
                      cudaStream_t stream, bool with_phi) {
    using F = typename C::F;
    if (!n) return;
    int mask = C::F::Params::kMontgomery ? 1 : 0;
    k_import_points<C><<<(n + 127) / 128, 128, 0, stream>>>(d_bytes, fmt, mask, n, reinterpret_cast<Affine<F>*>(d_points_out),
                                                           d_flags_out, nullptr);
    LAUNCHED();
    if constexpr (C::kGlv) {   // the endomorphism image right behind the table (PointTable::phi_off = n)
        if (with_phi) {
            k_phi_table<C><<<(n + 127) / 128, 128, 0, stream>>>(reinterpret_cast<const Affine<F>*>(d_points_out), n,
                                                               reinterpret_cast<F*>(reinterpret_cast<Affine<F>*>(d_points_out) + n));
            LAUNCHED();
        }
    }
    PORLA_CUDA(cudaGetLastError());
}

template <class C>
void import_impl(const uint8_t* d_bytes, int fmt, uint32_t n, PointTable* out, cudaStream_t stream) {
    using F = typename C::F;
    Affine<F>* pts = nullptr;
    uint8_t* flags = nullptr;
    uint32_t* d_count = nullptr;
    PORLA_CUDA(cudaMalloc(&pts, (size_t)(n ? n : 1) * (sizeof(Affine<F>) + (C::kGlv ? sizeof(F) : 0))));
    PORLA_CUDA(cudaMalloc(&flags, (size_t)(n ? n : 1)));
    PORLA_CUDA(cudaMalloc(&d_count, 4));
    PORLA_CUDA(cudaMemsetAsync(d_count, 0, 4, stream));
    if (n) {
        int mask = C::F::Params::kMontgomery ? 1 : 0;  // BN254: gnark flag bits in byte 0
        k_import_points<C><<<(n + 127) / 128, 128, 0, stream>>>(d_bytes, fmt, mask, n, pts, flags, d_count);
        LAUNCHED();
        if constexpr (C::kGlv) {
            k_phi_table<C><<<(n + 127) / 128, 128, 0, stream>>>(pts, n, reinterpret_cast<F*>(pts + n));
            LAUNCHED();
        }
        PORLA_CUDA(cudaGetLastError());
    }
    uint32_t h_count = 0;
    PORLA_CUDA(cudaMemcpyAsync(&h_count, d_count, 4, cudaMemcpyDeviceToHost, stream));
    PORLA_CUDA(cudaStreamSynchronize(stream));
    PORLA_CUDA(cudaFree(d_count));
    out->d_points = pts;
    out->n = n;
    out->n_inf = h_count;
    out->curve = CurveIdOf<C>::value;
    out->phi_off = C::kGlv ? n : 0u;
    out->d_phi_x = C::kGlv ? static_cast<void*>(pts + n) : nullptr;
    if (h_count == 0) {
        PORLA_CUDA(cudaFree(flags));
        out->d_flags = nullptr;
    } else {
        out->d_flags = flags;
    }
}

// ---------------------------------------------------------------------------- small / fixed-base MSMs: one launch
// plan.mode == kPlanBits: k_small_bits (plan.nwin = number of scalar bits, plan.c = 1);
// plan.mode == kPlanLut:  k_lut_sum over the table's look-up table (plan.nwin = 1).
template <class C>
void msm_small_impl(const PointTable& table, const uint8_t* d_scalars, uint32_t n, uint32_t nbatch, const MsmOptions& opt,
                    const MsmPlan& plan, uint8_t* d_out, void* d_out_xyzz, cudaStream_t stream) {
    using F = typename C::F;
    using XC = XYZZ<typename C::FC>;
    const bool lut = plan.mode == kPlanLut;
    const uint32_t slots = nbatch * (uint32_t)plan.nwin;
    uint32_t K = 1, nblk;
    if (lut) {
        // few MSMs: two table entries per thread, depth = log2 of the term count; many MSMs: one scalar
        // (all its windows) per thread, the machine is full anyway and the tree is 7 levels
        // few MSMs: two table entries per thread; many: whole scalars per thread, several of them once the machine
        // is full four times over, so that the block tree (7 levels, three of four warps idle) is paid less often
        uint32_t per_thread = 1;
        if (nbatch > 8) {
            const uint64_t want_threads = 148ull * 3 * kTreeThreads * 4;
            per_thread = (uint32_t)(((uint64_t)n * nbatch) / want_threads);
            if (per_thread < 1) per_thread = 1;
            if (per_thread > 16) per_thread = 16;
            while (per_thread > 1 && n / per_thread < (uint32_t)kTreeThreads) per_thread >>= 1;
        }
        K = nbatch > 8 ? (uint32_t)table.fb_nwin * per_thread : 2u;
        const uint32_t threads = (n * (uint32_t)table.fb_nwin + K - 1) / K;
        nblk = (threads + kTreeThreads - 1) / kTreeThreads;
    } else {
        nblk = (n + 2 * kTreeThreads - 1) / (2 * kTreeThreads);
    }
    if (!nblk) nblk = 1;
    const size_t need = Arena::padded((size_t)slots * nblk, sizeof(XYZZ<F>)) + Arena::padded(slots, 4) +
                        Arena::padded(slots, sizeof(XYZZ<F>)) + 1024;
    DeviceCtx& cx = device_ctx();
    Arena& g_arena = cx.arena;
    StageTimer& g_stage_timer = cx.timer;
    std::unique_lock<std::mutex> lock(cx.engine_mu, std::defer_lock);
    XYZZ<F>* partials;
    uint32_t* tickets;
    XYZZ<F>* wsum;
    if (opt.d_scratch && need <= opt.scratch_bytes) {   // caller's scratch: no shared state, no lock
        uint8_t* b = reinterpret_cast<uint8_t*>(opt.d_scratch);
        partials = reinterpret_cast<XYZZ<F>*>(b);
        b += Arena::padded((size_t)slots * nblk, sizeof(XYZZ<F>));
        tickets = reinterpret_cast<uint32_t*>(b);
        b += Arena::padded(slots, 4);
        wsum = reinterpret_cast<XYZZ<F>*>(b);
    } else {
        lock.lock();
        g_arena.acquire(stream);
        g_arena.reserve(need, stream);
        g_arena.reset();
        partials = g_arena.take<XYZZ<F>>((size_t)slots * nblk);
        tickets = g_arena.take<uint32_t>(slots);
        wsum = g_arena.take<XYZZ<F>>(slots);
    }
    for (int st = kStageCount; st <= kStageAccumulate; st++) g_stage_timer.mark(st, stream);
    if (nblk > 1) PORLA_CUDA(cudaMemsetAsync(tickets, 0, (size_t)slots * 4, stream));
    if (lut) {
        const int m_major = nbatch > 8 ? 1 : 0;
        k_lut_sum<C><<<m_major ? dim3(nbatch, nblk) : dim3(nblk, nbatch), kTreeThreads, 0, stream>>>(
            reinterpret_cast<const Affine<F>*>(table.d_lut), table.fb_c, table.fb_nwin, d_scalars, opt.scalar_be, n, K, m_major,
            partials, tickets, wsum);
    } else {
        k_small_bits<C><<<dim3(nblk, (uint32_t)plan.nwin, nbatch), kTreeThreads, 0, stream>>>(
            reinterpret_cast<const Affine<F>*>(table.d_points), table.d_flags, d_scalars, opt.scalar_be, n, opt.shared_points,
            partials, tickets, wsum);
    }
    LAUNCHED();
    g_stage_timer.mark(kStageReduce, stream);
    g_stage_timer.mark(kStageFinalize, stream);
    if (opt.d_window_sums) {
        PORLA_CUDA(cudaMemcpyAsync(opt.d_window_sums, wsum, (size_t)slots * sizeof(XYZZ<F>), cudaMemcpyDeviceToDevice, stream));
    } else {
        k_finalize<C><<<(nbatch + 31) / 32, 32, 0, stream>>>((const XC*)wsum, nbatch, plan.nwin, plan.c, opt.out_fmt, d_out,
                                                            reinterpret_cast<XC*>(d_out_xyzz));
        LAUNCHED();
    }
    g_stage_timer.mark(kNumStages, stream);
    if (lock.owns_lock()) g_arena.release(stream);
    PORLA_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------- the pipeline
// f(std::true_type) for a GLV MSM, else f(std::false_type): f launches the kernel instantiation decltype(g)::value selects,
// and curves without the endomorphism never instantiate the GLV one.
template <class C, class Fn>
void with_glv(bool glv, Fn&& f) {
    if constexpr (C::kGlv) {
        if (glv) {
            f(std::true_type{});
            return;
        }
    }
    f(std::false_type{});
}

template <class C>
void msm_impl(const PointTable& table, const uint8_t* d_scalars, uint32_t n, uint32_t nbatch,
                     const MsmOptions& opt, uint8_t* d_out, void* d_out_xyzz, cudaStream_t stream) {
    using F = typename C::F;
    const int curve = CurveIdOf<C>::value;
    {
        const MsmPlan plan = msm_plan_table(table, n, nbatch, opt);
        if (plan.mode != kPlanPipeline && n > 0) {
            msm_small_impl<C>(table, d_scalars, n, nbatch, opt, plan, d_out, d_out_xyzz, stream);
            return;
        }
    }
    MsmShape sh;
    sh.n = n;
    sh.nbatch = nbatch;
    sh.shared = opt.shared_points ? 1u : 0u;
    const bool streamed = opt.part_mode != kPartWhole;
    if (streamed && (nbatch != 1 || !opt.d_buckets || opt.window_bits <= 0 || opt.glv < 0 || !opt.no_fixed_base)) {
        fprintf(stderr, "[libmultiexp/porla_b200] FATAL: a streamed MSM part needs one MSM, a shared bucket array and a forced window layout\n");
        abort();
    }
    const bool fixed = table.fb_c > 0 && opt.shared_points && !opt.no_fixed_base &&
                       (opt.window_bits == 0 || opt.window_bits == table.fb_c);
    const MsmPlan wplan = fixed ? MsmPlan{table.fb_c, 1, kPlanPipeline, 0} : msm_plan(curve, n, nbatch, opt.window_bits, opt.glv);
    const bool glv = wplan.glv != 0;
    if (glv && !(C::kGlv && table.phi_off && table.d_phi_x)) {
        fprintf(stderr, "[libmultiexp/porla_b200] FATAL: GLV plan for a table without its endomorphism image\n");
        abort();
    }
    sh.c = wplan.c;
    sh.nwin = glv ? 2 * wplan.nwin : (C::kScalarBits + 1 + sh.c - 1) / sh.c;
    sh.nbuckets = 1u << (sh.c - 1);
    sh.fixed_n = fixed ? table.fb_n : 0u;
    sh.glv_wh = glv ? wplan.nwin : 0;
    sh.phi_off = glv ? table.phi_off : 0u;
    // window slots that own a bucket set: one per (msm, window) -- with GLV, per window of one half: window w of
    // k1 and window w of k2 fill the same buckets -- or one per msm in fixed-base mode
    const int slot_windows = fixed ? 1 : (glv ? wplan.nwin : sh.nwin);

    const uint64_t slots = (uint64_t)nbatch * slot_windows;
    const uint64_t nbt64 = slots * sh.nbuckets;
    const uint64_t pairs64 = (uint64_t)nbatch * n * sh.nwin;
    if (nbt64 >= (1ull << 32) || pairs64 >= (1ull << 32) || (uint64_t)nbatch * n >= (1ull << 31) ||
        (fixed && (uint64_t)table.fb_n * sh.nwin >= (1ull << 31))) {
        fprintf(stderr, "[libmultiexp/porla_b200] FATAL: MSM shape too large for 32-bit indexing\n");
        abort();
    }
    const uint32_t nbt = (uint32_t)nbt64;
    const uint32_t ntiles = (nbt + kScanTile - 1) / kScanTile;

    // reduction geometry: every thread pays a fixed ~17-addition weighting step on top of 2 additions per
    // bucket, so long chunks waste less work, but the kernel is latency-bound until the machine is full
    // (one dependent XYZZ addition is ~7 us on a lone warp).  Measured optimum (2^16 .. 2^22 points): about
    // 24 k threads in total; chunks of 4 .. 64 buckets.
    uint32_t chunk = 64;
    while (chunk > 4 && (uint64_t)nbt / chunk < 24576ull) chunk >>= 1;
    while (chunk > 4 && sh.nbuckets / chunk < 4) chunk >>= 1;
    if (const char* e = getenv("PORLA_REDUCE_CHUNK")) { if (atoi(e) >= 1) chunk = (uint32_t)atoi(e); }
    if (chunk > sh.nbuckets) chunk = sh.nbuckets;
    uint32_t threads_per_slot = (sh.nbuckets + chunk - 1) / chunk;  // nbuckets and chunk are powers of two
    uint32_t blocks_per_slot = (threads_per_slot + kRedThreads - 1) / kRedThreads;
    // Scan form on quads (k_reduce_scan + k_reduce_top: four lanes per point, 2.35 us per dependent addition instead of 6.9):
    // used while the reduction is bound by the depth of its additions, i.e. up to PORLA_REDUCE_QUAD_MAX buckets in total
    // (default C::kReduceQuadMax: 600 k for BN254, 300 k for secp256k1; above that k_reduce is near the multiplier pipe's limit and the quads' extra pipe work loses).  m = 2^log_m
    // buckets per quad: the smallest chunk that leaves at most PORLA_REDUCE_QUADS quads in flight (default 148 x 64: one block
    // of 64 quads, 8 warps, per SM), at most 64 and at least what keeps a slot within kTopMaxBlocks blocks.
    // PORLA_REDUCE_V1=1 keeps the round-1 kernel at every size.
    static const uint64_t quad_max = [] { const char* e = getenv("PORLA_REDUCE_QUAD_MAX"); return e ? (uint64_t)atoll(e) : (uint64_t)C::kReduceQuadMax; }();
    static const uint64_t quad_target = [] { const char* e = getenv("PORLA_REDUCE_QUADS"); return e && atoll(e) > 0 ? (uint64_t)atoll(e) : 148ull * kQuadsPerBlock; }();
    const bool reduce_v1 = getenv("PORLA_REDUCE_V1") != nullptr || (uint64_t)nbt > quad_max;
    uint32_t log_m = 0;
    while (log_m < 6 && ((uint64_t)nbt >> log_m) > quad_target) log_m++;
    while ((sh.nbuckets >> log_m) > (uint32_t)(kTopMaxBlocks * kQuadsPerBlock)) log_m++;
    while (log_m > 0 && (1u << log_m) > sh.nbuckets) log_m--;
    const uint32_t scan_tps = sh.nbuckets >> log_m;                                        // quads per slot
    const uint32_t scan_group = scan_tps >= (uint32_t)kQuadsPerBlock ? (uint32_t)kQuadsPerBlock : scan_tps;
    const uint32_t scan_bps = scan_tps >= (uint32_t)kQuadsPerBlock ? scan_tps / kQuadsPerBlock : 1u;   // blocks per slot
    if (!reduce_v1) blocks_per_slot = 2 * scan_bps;                                        // partials: out_w then out_s

    // accumulation geometry: slice length L (pairs per thread)
    const uint64_t pairs_cap = pairs64 ? pairs64 : 1;
    // One "wave" = the threads of k_accumulate resident at once (4 blocks x 128 threads per SM at 106
    // registers).  L is the slice length that fills a whole number of waves with slices of at most 64
    // pairs; small MSMs get one wave of short slices, never slices so short that stitching the cut
    // buckets costs more than the additions (L = 4 made a 2^16-point MSM spend 6x longer in k_stitch
    // than in k_accumulate).
    const uint64_t wave = 148ull * 4ull * kAccThreads;
    const uint64_t waves = (pairs_cap + wave * 64 - 1) / (wave * 64);
    uint32_t L = (uint32_t)((pairs_cap + waves * wave - 1) / (waves * wave));
    if (waves == 1) {
        // A single wave does better three quarters full with longer slices: 12 warps per SM already saturate the
        // multiplier pipe and every slice boundary saved is a partial sum less to stitch (measured: 2^16 terms,
        // 0.96 wave of 18-pair slices 0.353 ms, 0.72 wave of 24-pair slices 0.301 ms; 2^17: 0.560 -> 0.519 ms).
        const uint64_t l2 = pairs_cap / (wave * 18 / 25);
        if (l2 >= 16 && l2 <= 64) L = (uint32_t)l2;
    }
    if (L < 16) L = 16;
    if (L > 64) L = 64;
    if (const char* e = getenv("PORLA_SLICE_LEN")) { if (atoi(e) >= 2) L = (uint32_t)atoi(e); }
    const uint32_t nslices_cap = (uint32_t)((pairs_cap + L - 1) / L);
    // One serial XYZZ addition is ~7 us of latency: with few slices in flight (small MSMs) a bucket cut into
    // dozens of slices is better finished by a cooperating block; with the machine full, the serial loop in
    // every owner thread has the higher throughput (2^24, c = 20: 16 k top-window buckets of 17 slices).
    const uint32_t serial_limit = nslices_cap < 200000u ? kStitchSerialSmall : kStitchSerial;
    const uint32_t long_cap = (uint32_t)(pairs_cap / ((uint64_t)L * serial_limit)) + 2;

    // sort path: shared-memory radix partition (two MSD passes) for large single MSMs, else one returning
    // global atomic per pair
    const bool radix = nbatch == 1 && n >= (1u << 19) && sh.nwin <= 28 && sh.c >= 9 && sh.c <= 20 && (sh.nbuckets >> (sh.c / 2)) <= (uint32_t)kPartMaxBins && !getenv("PORLA_ATOMIC_SCATTER");
    const int lb = sh.c / 2;                                   // coarse bin = 2^lb consecutive buckets
    const uint32_t ncoarse = radix ? (nbt >> lb) : 0u;
    DeviceCtx& cx = device_ctx();
    Arena& g_arena = cx.arena;
    StageTimer& g_stage_timer = cx.timer;
    std::lock_guard<std::mutex> lock(cx.engine_mu);
    size_t need = (radix ? Arena::padded(pairs_cap, 8) + Arena::padded(ncoarse, 4) : 0) + Arena::padded(nbt, 4) * 2 + Arena::padded(ntiles + 1, 4) + 512 +
                  Arena::padded(pairs_cap, 8) + (streamed ? 0 : Arena::padded(nbt, sizeof(XYZZ<F>))) +
                  2 * Arena::padded(nslices_cap, sizeof(XYZZ<F>)) + Arena::padded(long_cap, 8) +
                  Arena::padded(slots * blocks_per_slot, sizeof(XYZZ<F>)) + Arena::padded(slots, sizeof(XYZZ<F>));
    g_arena.acquire(stream);
    g_arena.reserve(need, stream);
    g_arena.reset();
    uint32_t* counters = g_arena.take<uint32_t>(nbt);
    uint32_t* offsets = g_arena.take<uint32_t>(nbt);
    uint32_t* tile_sums = g_arena.take<uint32_t>(ntiles + 1);
    uint32_t* grand = g_arena.take<uint32_t>(1);       // total number of (point, window) pairs
    uint32_t* long_count = g_arena.take<uint32_t>(1);
    uint2* sorted = g_arena.take<uint2>(pairs_cap);
    uint2* part = radix ? g_arena.take<uint2>(pairs_cap) : nullptr;
    uint32_t* coarse_cursor = radix ? g_arena.take<uint32_t>(ncoarse) : nullptr;
    XYZZ<F>* buckets = streamed ? reinterpret_cast<XYZZ<F>*>(opt.d_buckets) : g_arena.take<XYZZ<F>>(nbt);
    const int into = opt.part_mode == kPartMiddle || opt.part_mode == kPartLast;
    XYZZ<F>* part_head = g_arena.take<XYZZ<F>>(nslices_cap);
    XYZZ<F>* part_tail = g_arena.take<XYZZ<F>>(nslices_cap);
    uint2* long_runs = g_arena.take<uint2>(long_cap);
    XYZZ<F>* partials = g_arena.take<XYZZ<F>>(slots * blocks_per_slot);
    XYZZ<F>* wsum = g_arena.take<XYZZ<F>>(slots);

    const Affine<F>* points = reinterpret_cast<const Affine<F>*>(fixed ? table.d_fb_points : table.d_points);
    // the cold kernels see the same records through the compact (outlined-multiply) field type
    using FC = typename C::FC;
    using XC = XYZZ<FC>;
    static_assert(sizeof(XC) == sizeof(XYZZ<F>), "layouts must coincide");
    const uint64_t total_scalars = (uint64_t)n * nbatch;

    g_stage_timer.mark(kStageCount, stream);
    // Radix path without the exact histogram (k_coarse_count ... k_fine_smem, msm_kernels.cuh): a coarse count places the coarse
    // bins, the coarse partition fills them, and ONE block per bin sorts it by bucket through shared memory.  Used when a bin is
    // expected to fit the block's shared memory (pairs / bins <= 0.95 kBigBin; bins that overflow on skewed inputs take the
    // tile-based route); PORLA_SORT_V2=0 / 1 forces.  Measured at 2^24 (ncu): exact count 1.55 -> coarse count 0.52 ms, fine pass
    // 2.07 -> see profiles/r02b_sort_without_exact_histogram.txt.
    const char* sv2 = getenv("PORLA_SORT_V2");
    const bool v2_fits = ncoarse > 0 && pairs_cap / ncoarse <= (uint64_t)(kBigBin * 0.95);
    const bool sort_v2 = radix && lb <= 10 && (size_t)ncoarse * 4 <= (size_t)kCoarseCountSmem && (sv2 ? sv2[0] == '1' : v2_fits);
    PORLA_CUDA(cudaMemsetAsync(counters, 0, (size_t)nbt * 4, stream));
    PORLA_CUDA(cudaMemsetAsync(grand, 0, 4, stream));
    PORLA_CUDA(cudaMemsetAsync(long_count, 0, 4, stream));
    // empty bucket = infinity: the whole array is cleared, except on the sort_v2 path, whose fine pass knows the empty buckets of
    // every coarse bin and clears just those (k_fine_smem / k_big_scan)
    static_assert(sizeof(XYZZ<F>) == 128, "k_fine_smem / k_big_scan clear 128-byte bucket records");
    if (!into && !sort_v2) PORLA_CUDA(cudaMemsetAsync(buckets, 0, (size_t)nbt * sizeof(XYZZ<F>), stream));
    uint4* zero_buckets = into ? nullptr : reinterpret_cast<uint4*>(buckets);
    if (radix) {
        static std::once_flag attr_once[kMaxDevices];   // function attributes are per device
        std::call_once(attr_once[current_device()], [] {
            PORLA_CUDA(cudaFuncSetAttribute(k_coarse_count<C, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kCoarseCountSmem));
            PORLA_CUDA(cudaFuncSetAttribute(k_partition_coarse<C, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPartCoarseSmem));
            if constexpr (C::kGlv) {
                PORLA_CUDA(cudaFuncSetAttribute(k_coarse_count<C, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kCoarseCountSmem));
                PORLA_CUDA(cudaFuncSetAttribute(k_partition_coarse<C, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPartCoarseSmem));
            }
            PORLA_CUDA(cudaFuncSetAttribute(k_partition_fine<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPartFineSmem));
            PORLA_CUDA(cudaFuncSetAttribute(k_partition_fine<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPartFineSmem));
            PORLA_CUDA(cudaFuncSetAttribute(k_fine_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, kFineLocalSmem));
        });
    }
    if (total_scalars && sort_v2) {
        uint32_t* coarse_count = offsets;                 // the exact-offset array is not needed on this path: reuse it
        uint32_t* coarse_off = offsets + ncoarse + 1;     // (nbt >= 2 * (ncoarse + 1): 2^lb >= 16 buckets per bin)
        PORLA_CUDA(cudaMemsetAsync(coarse_count, 0, (size_t)(ncoarse + 1) * 4, stream));
        uint32_t cgrid = (uint32_t)((total_scalars + kCoarseCountThreads - 1) / kCoarseCountThreads);
        if (cgrid > 148u * 2u) cgrid = 148u * 2u;
        with_glv<C>(glv, [&](auto g) {
            k_coarse_count<C, decltype(g)::value><<<cgrid, kCoarseCountThreads, (size_t)ncoarse * 4, stream>>>(
                d_scalars, opt.scalar_be, table.d_flags, sh, lb, ncoarse, coarse_count);
        });
        LAUNCHED();
        g_stage_timer.mark(kStageScan, stream);
        k_coarse_scan<<<1, 1024, 0, stream>>>(coarse_count, ncoarse, coarse_off, coarse_cursor, grand);
        LAUNCHED();
        g_stage_timer.mark(kStageScatter, stream);
        with_glv<C>(glv, [&](auto g) {
            k_partition_coarse<C, decltype(g)::value><<<(n + kPartTile - 1) / kPartTile, kPartThreads, kPartCoarseSmem, stream>>>(
                d_scalars, opt.scalar_be, table.d_flags, sh, lb, coarse_cursor, part);
        });
        LAUNCHED();
        k_fine_smem<<<ncoarse, kFineSmemThreads, kFineLocalSmem, stream>>>(part, coarse_off, lb, sorted, zero_buckets);
        LAUNCHED();
        // bins too long for one block (skewed inputs): counted, scanned and scattered by tiles; no-ops otherwise
        const uint32_t tiles = (uint32_t)((pairs_cap + kFineTile - 1) / kFineTile);
        k_big_count<<<tiles, kFineThreads, 0, stream>>>(part, grand, coarse_off, lb, counters);
        LAUNCHED();
        k_big_scan<<<ncoarse, kFineLocalThreads, 0, stream>>>(coarse_off, lb, counters, zero_buckets);
        LAUNCHED();
        k_partition_fine<true><<<tiles, kFineThreads, kPartFineSmem, stream>>>(part, grand, coarse_off, lb, counters, sorted);
        LAUNCHED();
    } else if (total_scalars) {
        uint32_t grid = (uint32_t)((total_scalars + 255) / 256);
        if (grid > 148u * 32u) grid = 148u * 32u;
        with_glv<C>(glv, [&](auto g) {
            k_digits<C, false, decltype(g)::value><<<grid, 256, 0, stream>>>(d_scalars, opt.scalar_be, table.d_flags, sh, 0, sh.nwin,
                                                                              counters, nullptr);
        });
        LAUNCHED();
        g_stage_timer.mark(kStageScan, stream);
        k_scan_tiles<<<ntiles, kScanThreads, 0, stream>>>(counters, offsets, nbt, tile_sums);
        LAUNCHED();
        k_scan_sums<<<1, kScanThreads, 0, stream>>>(tile_sums, ntiles, grand);
        LAUNCHED();
        k_scan_add<<<ntiles, kScanThreads, 0, stream>>>(offsets, counters, nbt, tile_sums);
        LAUNCHED();
        g_stage_timer.mark(kStageScatter, stream);
        if (radix) {
            k_init_coarse<<<(ncoarse + 255) / 256, 256, 0, stream>>>(offsets, nbt, lb, ncoarse, coarse_cursor);
            LAUNCHED();
            with_glv<C>(glv, [&](auto g) {
                k_partition_coarse<C, decltype(g)::value><<<(n + kPartTile - 1) / kPartTile, kPartThreads, kPartCoarseSmem, stream>>>(
                    d_scalars, opt.scalar_be, table.d_flags, sh, lb, coarse_cursor, part);
            });
            LAUNCHED();
            k_partition_fine<false><<<(uint32_t)((pairs_cap + kFineTile - 1) / kFineTile), kFineThreads, kPartFineSmem, stream>>>(
                part, grand, nullptr, lb, counters, sorted);
            LAUNCHED();
        } else {
        // windows per scatter launch: keep the written region of `sorted` (8 B per pair) around 64 MB
        int wgroup = sh.nwin;
        if (nbatch == 1) {
            uint64_t per_window = (uint64_t)n * 8;
            wgroup = (int)((64ull << 20) / (per_window ? per_window : 1));
            if (wgroup < 1) wgroup = 1;
            if (wgroup > sh.nwin) wgroup = sh.nwin;
        }
        for (int w0 = 0; w0 < sh.nwin; w0 += wgroup) {
            int w1 = w0 + wgroup < sh.nwin ? w0 + wgroup : sh.nwin;
            with_glv<C>(glv, [&](auto g) {
                k_digits<C, true, decltype(g)::value><<<grid, 256, 0, stream>>>(d_scalars, opt.scalar_be, table.d_flags, sh, w0, w1,
                                                                                 counters, sorted);
            });
            LAUNCHED();
        }
        }
    }
    if (total_scalars) {
        g_stage_timer.mark(kStageAccumulate, stream);
        k_accumulate<C><<<(nslices_cap + kAccThreads - 1) / kAccThreads, kAccThreads, 0, stream>>>(
            points, reinterpret_cast<const F*>(table.d_phi_x), sh.phi_off, sorted, grand, L, buckets, part_head, part_tail, into);
        LAUNCHED();
        k_stitch<C><<<(nslices_cap + 63) / 64, 64, 0, stream>>>(sorted, grand, L, buckets, part_head, part_tail, long_count,
                                                               long_runs, serial_limit);
        LAUNCHED();
        k_stitch_long<C><<<148, kLongThreads, 0, stream>>>(sorted, grand, L, (XC*)buckets, (const XC*)part_head, long_count,
                                                          long_runs);
        LAUNCHED();
    } else {
        g_stage_timer.mark(kStageScan, stream);
        g_stage_timer.mark(kStageScatter, stream);
        g_stage_timer.mark(kStageAccumulate, stream);
    }
    g_stage_timer.mark(kStageReduce, stream);
    if (opt.part_mode == kPartFirst || opt.part_mode == kPartMiddle) {   // the last part reduces the shared buckets
        g_stage_timer.mark(kStageFinalize, stream);
        g_stage_timer.mark(kNumStages, stream);
        g_arena.release(stream);
        PORLA_CUDA(cudaGetLastError());
        return;
    }
    if (slots * blocks_per_slot >= (1ull << 31)) {
        fprintf(stderr, "[libmultiexp/porla_b200] FATAL: too many window slots for one launch\n");
        abort();
    }
    const XYZZ<F>* window_sums = partials;
    if (reduce_v1) {
        const uint32_t rgrid = threads_per_slot >= (uint32_t)kRedThreads
                                   ? (uint32_t)(slots * blocks_per_slot)
                                   : (uint32_t)((slots + kRedThreads / threads_per_slot - 1) / (kRedThreads / threads_per_slot));
        k_reduce<C><<<rgrid, kRedThreads, 0, stream>>>((const XC*)buckets, sh.nbuckets, chunk, threads_per_slot, (uint32_t)slots,
                                                       (XC*)partials);
        LAUNCHED();
        if (blocks_per_slot > 1) {
            k_window_sums<C><<<(uint32_t)slots, kRedThreads, 0, stream>>>((const XC*)partials, blocks_per_slot, (XC*)wsum);
            LAUNCHED();
            window_sums = wsum;
        }
    } else {
        XYZZ<F>* out_w = partials;
        XYZZ<F>* out_s = out_w + slots * scan_bps;
        const uint32_t sgrid = scan_group == (uint32_t)kQuadsPerBlock
                                   ? (uint32_t)(slots * scan_bps)
                                   : (uint32_t)((slots + kQuadsPerBlock / scan_group - 1) / (kQuadsPerBlock / scan_group));
        k_reduce_scan<C><<<sgrid, kQuadThreads, 0, stream>>>(buckets, sh.nbuckets, log_m, scan_group, (uint32_t)slots, out_w, out_s);
        LAUNCHED();
        if (scan_bps > 1) {
            uint32_t log_u = log_m;                      // weight of one block: m * kQuadsPerBlock buckets
            while ((1u << log_u) < ((uint32_t)kQuadsPerBlock << log_m)) log_u++;
            k_reduce_top<C><<<(uint32_t)slots, kQuadThreads, 0, stream>>>(out_w, out_s, scan_bps, log_u, wsum);
            LAUNCHED();
            window_sums = wsum;
        }
    }
    g_stage_timer.mark(kStageFinalize, stream);
    if (opt.d_window_sums) {
        PORLA_CUDA(cudaMemcpyAsync(opt.d_window_sums, window_sums, slots * sizeof(XYZZ<F>), cudaMemcpyDeviceToDevice, stream));
    } else {
        k_finalize<C><<<(nbatch + 31) / 32, 32, 0, stream>>>((const XC*)window_sums, nbatch, slot_windows, sh.c, opt.out_fmt, d_out,
                                                            reinterpret_cast<XC*>(d_out_xyzz));
        LAUNCHED();
    }
    g_stage_timer.mark(kNumStages, stream);
    g_arena.release(stream);
    PORLA_CUDA(cudaGetLastError());
}

template <class C>
void precompute_impl(PointTable* t, int c, cudaStream_t stream) {
    using FC = typename C::FC;
    const int nwin = (C::kScalarBits + 1 + c - 1) / c;
    if (t->d_fb_points) PORLA_CUDA(cudaFree(t->d_fb_points));
    void* out = nullptr;
    PORLA_CUDA(cudaMalloc(&out, (size_t)nwin * (t->n ? t->n : 1) * sizeof(Affine<FC>)));
    if (t->n) {
        k_precompute_windows<C><<<(t->n + 127) / 128, 128, 0, stream>>>(reinterpret_cast<const Affine<FC>*>(t->d_points), t->n, c, nwin,
                                                                      reinterpret_cast<Affine<FC>*>(out));
        LAUNCHED();
        PORLA_CUDA(cudaGetLastError());
    }
    t->d_fb_points = out;
    t->fb_c = c;
    t->fb_nwin = nwin;
    t->fb_n = t->n;
    if (t->d_lut) PORLA_CUDA(cudaFree(t->d_lut));
    t->d_lut = nullptr;
}

// Look-up table of every window multiple (k_lut_build) on top of the fixed-base expansion.
template <class C>
void lut_impl(PointTable* t, cudaStream_t stream) {
    using FC = typename C::FC;
    if (!t->n || !t->d_fb_points) return;
    void* out = nullptr;
    const size_t entries = ((size_t)t->fb_nwin * t->n) << (t->fb_c - 1);
    PORLA_CUDA(cudaMalloc(&out, entries * sizeof(Affine<FC>)));
    const uint32_t threads = t->n * (uint32_t)t->fb_nwin;
    k_lut_build<C><<<(threads + 127) / 128, 128, 0, stream>>>(reinterpret_cast<const Affine<FC>*>(t->d_fb_points), t->d_flags, t->n,
                                                             t->fb_c, t->fb_nwin, reinterpret_cast<Affine<FC>*>(out));
    LAUNCHED();
    PORLA_CUDA(cudaGetLastError());
    t->d_lut = out;
}

template <class C>
void combine_impl(const void* d_parts, uint32_t count, uint32_t nbatch, int out_fmt, uint8_t* d_out, cudaStream_t stream) {
    using F = typename C::FC;
    k_combine<C><<<(nbatch + 63) / 64, 64, 0, stream>>>(reinterpret_cast<const XYZZ<F>*>(d_parts), count, nbatch, out_fmt, d_out);
    LAUNCHED();
    PORLA_CUDA(cudaGetLastError());
}

template <class C>
void scalar_mul_impl(const PointTable& table, const uint8_t* d_scalars, int scalar_be, uint32_t n, void* d_out_affine,
                     cudaStream_t stream) {
    using F = typename C::FC;
    k_scalar_mul<C><<<(n + 127) / 128, 128, 0, stream>>>(reinterpret_cast<const Affine<F>*>(table.d_points), table.n, d_scalars,
                                                        scalar_be, n, reinterpret_cast<Affine<F>*>(d_out_affine));
    LAUNCHED();
    PORLA_CUDA(cudaGetLastError());
}

template <class C>
void fixed_base_mul_impl(const PointTable& table, const uint8_t* d_scalars, int scalar_be, uint32_t n, int out_fmt,
                         uint8_t* d_out, cudaStream_t stream) {
    using F = typename C::F;
    const Affine<F>* lut = reinterpret_cast<const Affine<F>*>(table.d_lut);
    const uint32_t grid = (n + kFixedBaseThreads - 1) / kFixedBaseThreads;
    k_fixed_base_mul<C><<<grid, kFixedBaseThreads, 0, stream>>>(lut, table.fb_c, table.fb_nwin, d_scalars, scalar_be, n, out_fmt,
                                                                d_out);
    LAUNCHED();
    PORLA_CUDA(cudaGetLastError());
}

template <class C>
void butterfly_impl(PointTable* t, uint32_t m, const uint8_t* d_twiddles, int scalar_be, cudaStream_t stream) {
    const uint32_t nb = t->n / 2;
    if (!nb) return;
    if (!t->d_flags) {   // outputs may be infinity (A0 = +-t): from now on the table carries flags
        PORLA_CUDA(cudaMalloc(&t->d_flags, t->n));
        PORLA_CUDA(cudaMemsetAsync(t->d_flags, 0, t->n, stream));
    }
    // Measured per stage (one B200, warm clocks), BN254:
    //   n = 1024 (512 butterflies, pure latency): plain double-and-add 2.16 ms inlined / 2.69 ms compact field type;
    //            GLV joint double-and-add (127 doublings, one extra inversion per butterfly) 1.39 / 1.67 ms
    //   n = 2^20: plain 42.1 / 47.3 ms, GLV 26.6 / 31.3 ms
    // so both curves run the GLV forms on the inlined type.  secp256k1 (profiles/r04_secp_butterfly_times.txt): the compact
    // type no longer pays off once the GLV form halves the doublings (2.720 / 5.500 ms against 2.717 / 5.396 ms inlined at
    // 65 536 / 131 072 butterflies).
    // Few butterflies (C::kButterflyQuadMax): four lanes per butterfly (k_butterfly_quad; PORLA_BUTTERFLY_QUAD=0 / 1 forces).
    auto* pf = reinterpret_cast<Affine<typename C::F>*>(t->d_points);
    const dim3 grid((nb + 127) / 128);
    const char* fq = getenv("PORLA_BUTTERFLY_QUAD");
    if (fq ? fq[0] == '1' : nb <= C::kButterflyQuadMax) {
        k_butterfly_quad<C><<<(nb * 4 + kBflyQuadThreads - 1) / kBflyQuadThreads, kBflyQuadThreads, 0, stream>>>(pf, t->d_flags, t->n, m, d_twiddles, scalar_be);
    } else {
        k_butterfly<C, typename C::F><<<grid, 128, 0, stream>>>(pf, t->d_flags, t->n, m, d_twiddles, scalar_be);
    }
    LAUNCHED();
    if constexpr (C::kGlv) {
        if (t->phi_off) {   // the points changed: so does their endomorphism image
            k_phi_table<C><<<(t->n + 127) / 128, 128, 0, stream>>>(reinterpret_cast<const Affine<typename C::F>*>(t->d_points), t->n,
                                                                  reinterpret_cast<typename C::F*>(t->d_phi_x));
            LAUNCHED();
        }
    }
    PORLA_CUDA(cudaGetLastError());
}

template <class C>
void align_scalars_impl(uint32_t* d_data, uint32_t total, uint8_t* d_scalars_be, cudaStream_t stream) {
    if (!total) return;
    k_align_scalars<C><<<(total + 127) / 128, 128, 0, stream>>>(d_data, total, d_scalars_be);
    LAUNCHED();
    PORLA_CUDA(cudaGetLastError());
}

template <class C>
void audit_aggregate_impl(const uint32_t* d_coefs, const uint32_t* d_blocks, uint32_t n, uint32_t chunks, uint8_t* d_b_mod_be,
                          uint8_t* d_c_be, cudaStream_t stream) {
    if (!chunks) return;
    k_audit_aggregate<C><<<chunks, kAggThreads, 0, stream>>>(d_coefs, d_blocks, n, chunks, d_b_mod_be, d_c_be);
    LAUNCHED();
    PORLA_CUDA(cudaGetLastError());
}

inline void data_butterfly_impl(uint32_t* d_blocks, uint32_t n_blocks, uint32_t chunks, uint32_t m, const uint8_t* d_twiddles,
                                const DataFftParams& prm, cudaStream_t stream) {
    const uint64_t total = (uint64_t)(n_blocks / 2) * chunks;
    if (!total) return;
    k_data_butterfly<<<(uint32_t)((total + 127) / 128), 128, 0, stream>>>(d_blocks, n_blocks, chunks, m, d_twiddles, prm);
    LAUNCHED();
    PORLA_CUDA(cudaGetLastError());
}

template <class C>
void export_impl(const void* d_affine, uint32_t n, int fmt, uint8_t* d_out, cudaStream_t stream) {
    using F = typename C::F;
    k_export_points<C><<<(n + 127) / 128, 128, 0, stream>>>(reinterpret_cast<const Affine<F>*>(d_affine), n, fmt, d_out);
    LAUNCHED();
    PORLA_CUDA(cudaGetLastError());
}

template <class C>
void field_mul_impl(const void* d_a, const void* d_b, uint32_t n, int op, void* d_out, cudaStream_t stream) {
    using F = typename C::F;
    k_field_mul<C><<<(n + 127) / 128, 128, 0, stream>>>(reinterpret_cast<const F*>(d_a), reinterpret_cast<const F*>(d_b), n, op,
                                                       reinterpret_cast<F*>(d_out));
    LAUNCHED();
    PORLA_CUDA(cudaGetLastError());
}

#define PORLA_INSTANTIATE_CURVE(C)                                                                                     \
    template void import_impl<C>(const uint8_t*, int, uint32_t, PointTable*, cudaStream_t);                            \
    template void import_into_impl<C>(const uint8_t*, int, uint32_t, void*, uint8_t*, cudaStream_t, bool);             \
    template void msm_impl<C>(const PointTable&, const uint8_t*, uint32_t, uint32_t, const MsmOptions&, uint8_t*,      \
                              void*, cudaStream_t);                                                                    \
    template void combine_impl<C>(const void*, uint32_t, uint32_t, int, uint8_t*, cudaStream_t);                       \
    template void precompute_impl<C>(PointTable*, int, cudaStream_t);                                                  \
    template void lut_impl<C>(PointTable*, cudaStream_t);                                                              \
    template void scalar_mul_impl<C>(const PointTable&, const uint8_t*, int, uint32_t, void*, cudaStream_t);           \
    template void fixed_base_mul_impl<C>(const PointTable&, const uint8_t*, int, uint32_t, int, uint8_t*, cudaStream_t); \
    template void export_impl<C>(const void*, uint32_t, int, uint8_t*, cudaStream_t);                                  \
    template void butterfly_impl<C>(PointTable*, uint32_t, const uint8_t*, int, cudaStream_t);                         \
    template void align_scalars_impl<C>(uint32_t*, uint32_t, uint8_t*, cudaStream_t);                                  \
    template void audit_aggregate_impl<C>(const uint32_t*, const uint32_t*, uint32_t, uint32_t, uint8_t*, uint8_t*,    \
                                          cudaStream_t);                                                               \
    template void field_mul_impl<C>(const void*, const void*, uint32_t, int, void*, cudaStream_t);

}  // namespace porla
