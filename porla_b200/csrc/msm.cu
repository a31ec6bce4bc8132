// Curve-independent host infrastructure and the curve dispatchers of the device MSM engine.
// The templated drivers live in msm_impl.cuh (instantiated in msm_bn254.cu / msm_secp.cu).
#include "msm.h"

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <cstring>

#include "arena.h"
#include "ec.cuh"
#include "host_fp64.hpp"

namespace porla {

std::atomic<uint64_t> g_launches{0};
uint64_t launches_issued() { return g_launches.load(); }

void cuda_check(cudaError_t e, const char* what, const char* file, int line) {
    if (e == cudaSuccess) return;
    fprintf(stderr, "[libmultiexp/porla_b200] FATAL CUDA error %d (%s) at %s:%d in %s\n", (int)e,
            cudaGetErrorString(e), file, line, what);
    fprintf(stderr, "[libmultiexp/porla_b200] this library has no CPU fallback; a B200 (sm_100a) is required\n");
    abort();
}

static std::once_flag g_dev_once;
static int g_device = -1;
static int g_device_count = 0;
static bool g_device_pinned = false;
static thread_local int t_device = -1;    // >= 0 while the thread holds a DeviceScope

bool device_available() {
    int count = 0;
    return cudaGetDeviceCount(&count) == cudaSuccess && count > 0;
}

int device_count() {
    int count = 0;
    return cudaGetDeviceCount(&count) == cudaSuccess ? count : 0;
}

static void device_init_once() {
    std::call_once(g_dev_once, [] {
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0) {
            fprintf(stderr,
                    "[libmultiexp/porla_b200] FATAL: no CUDA device (%s); the MSM path is GPU-only, "
                    "there is no CPU fallback\n",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
            abort();
        }
        if (count > kMaxDevices) count = kMaxDevices;
        int dev = 0;
        const char* s = getenv("PORLA_DEVICE");
        if (!s) s = getenv("LOCAL_RANK");
        if (s) {
            dev = atoi(s) % count;
            g_device_pinned = true;
        }
        g_device_count = count;
        g_device = dev;
    });
}

// stream-ordered allocations (twiddle / result staging of the batched entry points) stay in the pool
// between calls: with the default threshold of 0 every synchronize hands the memory back to the driver
// and the next call pays a real allocation (milliseconds of jitter on a 2 ms butterfly stage)
static void device_first_use(int dev) {
    static std::once_flag once[kMaxDevices];
    std::call_once(once[dev], [dev] {
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            uint64_t keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    });
}

int device_init() {
    device_init_once();
    const int dev = t_device >= 0 ? t_device : g_device;
    PORLA_CUDA(cudaSetDevice(dev));
    device_first_use(dev);
    return dev;
}

int default_device() {
    device_init_once();
    return g_device;
}

int current_device() {
    device_init_once();
    return t_device >= 0 ? t_device : g_device;
}

bool device_pinned_by_env() {
    device_init_once();
    return g_device_pinned;
}

DeviceScope::DeviceScope(int dev) {
    device_init_once();
    if (dev < 0 || dev >= g_device_count) {
        fprintf(stderr, "[libmultiexp/porla_b200] FATAL: device %d outside the %d visible devices\n", dev, g_device_count);
        abort();
    }
    prev = t_device;
    t_device = dev;
    PORLA_CUDA(cudaSetDevice(dev));
    device_first_use(dev);
}
DeviceScope::~DeviceScope() {
    t_device = prev;
    cudaSetDevice(prev >= 0 ? prev : g_device);
}

static DeviceCtx g_ctx[kMaxDevices];
DeviceCtx& device_ctx() {
    device_init_once();
    return g_ctx[t_device >= 0 ? t_device : g_device];
}

// Stage timing is switched on for the whole process; every device records its own events and the read-out is that
// of the calling thread's device.
static bool g_stage_timing = false;
void stage_timing_enable(int on) {
    g_stage_timing = on != 0;
    for (auto& c : g_ctx) c.timer.enabled = g_stage_timing;
}
int stage_timing_read(float* ms_out) {
    StageTimer& tm = device_ctx().timer;
    if (!tm.enabled || !tm.created) return 0;
    PORLA_CUDA(cudaEventSynchronize(tm.ev[kNumStages]));
    for (int i = 0; i < kNumStages; i++) {
        float ms = 0;
        // a stage that was skipped (empty MSM) keeps a stale event: report what CUDA gives
        if (cudaEventElapsedTime(&ms, tm.ev[i], tm.ev[i + 1]) != cudaSuccess) ms = 0;
        ms_out[i] = ms;
    }
    return kNumStages;
}

template <class C> void import_impl(const uint8_t*, int, uint32_t, PointTable*, cudaStream_t);
template <class C> void import_into_impl(const uint8_t*, int, uint32_t, void*, uint8_t*, cudaStream_t, bool);
template <class C> void msm_impl(const PointTable&, const uint8_t*, uint32_t, uint32_t, const MsmOptions&, uint8_t*, void*, cudaStream_t);
template <class C> void precompute_impl(PointTable*, int, cudaStream_t);
template <class C> void lut_impl(PointTable*, cudaStream_t);
constexpr uint32_t kLutMaxBases = 2048;   // 512 MiB of table at most
constexpr uint32_t kLutMaxBasesBatched = 8192;
constexpr int kLutWindow = 8;
template <class C> void combine_impl(const void*, uint32_t, uint32_t, int, uint8_t*, cudaStream_t);
template <class C> void scalar_mul_impl(const PointTable&, const uint8_t*, int, uint32_t, void*, cudaStream_t);
template <class C> void fixed_base_mul_impl(const PointTable&, const uint8_t*, int, uint32_t, int, uint8_t*, cudaStream_t);
template <class C> void export_impl(const void*, uint32_t, int, uint8_t*, cudaStream_t);
template <class C> void butterfly_impl(PointTable*, uint32_t, const uint8_t*, int, cudaStream_t);
template <class C> void align_scalars_impl(uint32_t*, uint32_t, uint8_t*, cudaStream_t);
template <class C> void audit_aggregate_impl(const uint32_t*, const uint32_t*, uint32_t, uint32_t, uint8_t*, uint8_t*, cudaStream_t);
template <class C> void field_mul_impl(const void*, const void*, uint32_t, int, void*, cudaStream_t);

#define DISPATCH(curve, fn, ...)                                  \
    do {                                                          \
        if ((curve) == kCurveBn254) fn<Bn254>(__VA_ARGS__);       \
        else fn<Secp256k1>(__VA_ARGS__);                          \
    } while (0)

// ---------------------------------------------------------------------------- window choice
static int scalar_bits(int curve) { return curve == kCurveBn254 ? Bn254::kScalarBits : Secp256k1::kScalarBits; }

// Cost of one bucket in the reduction, in units of one bucket-accumulation mixed addition
// (measured: k_stitch + k_reduce time per bucket / k_accumulate time per pair).
static double bucket_cost() {
    static const double v = [] {
        const char* e = getenv("PORLA_BUCKET_COST");
        return e && atof(e) > 0 ? atof(e) : 4.0;
    }();
    return v;
}

// Cost (in bucket-accumulation mixed additions) of running `terms` terms of `bits`-bit scalars per MSM with
// window size c; < 0 when c is not usable.
static double window_cost(int bits, double terms, uint32_t nbatch, int c) {
    int nwin = (bits + 1 + c - 1) / c;
    double nb = (double)(1u << (c - 1));
    // one mixed add per (point, window); ~4 mixed-add equivalents per bucket in the reduction
    double cost = (double)nwin * (terms + bucket_cost() * nb);
    double total_buckets = (double)nbatch * nwin * nb;
    if (total_buckets > 3.0e9) return -1;           // 32-bit bucket ids
    if (total_buckets * 128.0 > 48.0e9) return -1;  // bucket array budget
    // A window size that leaves only a few bits for the top window puts n / 2^(t-1) points into each
    // of its few buckets: contended counters in the sort and long serial stitches in the accumulation
    // (measured at 2^18: c = 13 -> 1.99 ms, c = 15 -> 1.33 ms; secp256k1 2^18: c = 13 -> 1.38 ms,
    // c = 16 -> 1.23 ms).  Skip such sizes once the load matters, penalise them mildly below that.  A top
    // window that still has more than 2^10 buckets spreads the load over enough threads (c = 20).
    int t_top = bits + 1 - (nwin - 1) * c;
    if (t_top < c - 1 && t_top <= 10) {
        uint64_t load_top = (uint64_t)terms >> (t_top > 1 ? t_top - 1 : 0);
        if (load_top > 1024) return -1;
        if (load_top > 256) cost *= 1.15;
    }
    // Buckets much longer than a slice (64 pairs) are cut into many partial sums that one owner thread
    // per bucket adds serially while its warp idles (2^26: c = 17 -> 225 ms, c = 20 -> 168 ms).
    cost *= 1.0 + 0.02 * (terms / nb) / 64.0;
    return cost;
}

static bool glv_allowed(int curve) {
    return curve == kCurveBn254 && Bn254::kGlv && !getenv("PORLA_NO_GLV");
}

// Window size and whether to split the scalars with the GLV endomorphism (BN254): 2n terms of 127-bit scalars need
// half as many windows, hence half as many buckets to reduce, for the same number of bucket updates whenever
// ceil(128/c) * 2 == ceil(255/c) (c = 16: 8 + 8 windows instead of 16).  forced_c > 0 fixes the window size.
struct WindowChoice {
    int c;
    int glv;
};
static WindowChoice choose_window_ex(int curve, uint32_t n, uint32_t nbatch, int forced_c, int forced_glv = -1) {
    const char* env = getenv("PORLA_WINDOW_BITS");
    if (forced_c <= 0 && env && atoi(env) >= 2 && atoi(env) <= 24) forced_c = atoi(env);
    const int bits = scalar_bits(curve);
    const bool glv_ok = glv_allowed(curve);
    const char* force_glv = getenv("PORLA_GLV");
    // a plan code fixes the whole layout, whatever the window size (the search below only covers 3 .. 20)
    if (forced_c > 0 && forced_glv == 1 && glv_ok) return WindowChoice{forced_c, 1};
    if (forced_c > 0 && forced_glv == 0) return WindowChoice{forced_c, 0};
    double best = 1e300;
    WindowChoice ch{forced_c > 0 ? forced_c : 4, 0};
    for (int c = 3; c <= 20; c++) {   // 20: the widest window the shared-memory radix partition packs
        if (forced_c > 0 && c != forced_c) continue;
        double plain = window_cost(bits, (double)n, nbatch, c);
        if (force_glv && force_glv[0] == '1' && glv_ok) plain = -1;
        if (plain >= 0 && plain < best) {
            best = plain;
            ch = WindowChoice{c, 0};
        }
        // measured (one B200): 2^16 c = 13 0.77 -> 0.70 ms, 2^18 1.32 -> 1.29 ms, 2^20 c = 16 3.62 -> 3.53 ms; the
        // wide windows the model would pick at 2^22 (c = 19, 7 windows per half) lose to the plain c = 17
        // (12.4 against 11.8 ms: 1.8 M buckets to reduce), so the split is offered up to c = 16 only
        if (glv_ok && (c <= 16 || forced_c > 0)) {
            double split = window_cost(Bn254::kGlvBits, 2.0 * (double)n, nbatch, c);
            if (split >= 0 && split < best) {
                best = split;
                ch = WindowChoice{c, 1};
            }
        }
    }
    return ch;
}

int choose_window(int curve, uint32_t n, uint32_t nbatch) { return choose_window_ex(curve, n, nbatch, 0).c; }

int choose_window_fixed_base(int curve, uint32_t n, uint32_t nbatch) {
    const int bits = scalar_bits(curve);
    double best = 1e300;
    int best_c = 8;
    for (int c = 4; c <= 20; c++) {   // 20: the widest window the shared-memory radix partition packs (measured: 2^24 with
                                      // c = 22 45.1 ms against 43.5 ms for the general path, c = 20 ~39 ms)
        int nwin = (bits + 1 + c - 1) / c;
        double nb = (double)(1u << (c - 1));
        double cost = (double)nwin * (double)n + 4.0 * nb;   // one shared bucket set per MSM
        if ((double)nbatch * nb * 128.0 > 48.0e9) continue;
        if ((double)nwin * (double)n >= 2.0e9) continue;
        int t_top = bits + 1 - (nwin - 1) * c;   // see choose_window: the short top window's digits pile up in a few buckets
        if (t_top < c - 1 && t_top <= 10 && ((uint64_t)n >> (t_top > 1 ? t_top - 1 : 0)) > 1024) continue;
        if (cost < best) {
            best = cost;
            best_c = c;
        }
    }
    return best_c;
}

int table_precompute(PointTable* t, int c, uint32_t n_hint, uint32_t batch_hint, cudaStream_t stream) {
    device_init();
    // Small tables (Porla's 128-point SRS / generator sets) get the full look-up table of window multiples with
    // 8-bit windows: 32 windows x 128 multiples x 64 B = 256 KiB per base, L2-resident for 128 bases.  A table
    // shared by a large batch (BASELINE config 3: 4096 commitments over 4096 bases) gets the WIDEST windows whose
    // table fits the HBM budget (c = 15: 17 windows x 16384 multiples x 4096 bases x 64 B = 73 GB of the B200's
    // 180 GB): every scalar then costs 17 gathers and mixed additions, with no sort and no bucket reduction.
    bool want_lut = false;
    if (c <= 0 && t->n > 0 && t->n <= kLutMaxBasesBatched && (uint64_t)(n_hint ? n_hint : t->n) * (batch_hint ? batch_hint : 1) >= (1ull << 22) &&
        !getenv("PORLA_NO_LUT")) {
        const char* e = getenv("PORLA_LUT_BUDGET_GB");
        double budget = (e && atof(e) > 0 ? atof(e) : 80.0) * 1e9;
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && (double)free_b * 0.6 < budget) budget = (double)free_b * 0.6;
        const int bits = scalar_bits(t->curve);
        for (int cc = 16; cc >= 9; cc--) {
            const double nwin = (double)((bits + 1 + cc - 1) / cc);
            if (nwin * (double)t->n * (double)(1u << (cc - 1)) * 64.0 <= budget) {
                c = cc;
                want_lut = true;
                break;
            }
        }
    }
    if (c <= 0 && t->n > 0 && t->n <= kLutMaxBases && !getenv("PORLA_NO_LUT")) {
        c = kLutWindow;
        want_lut = true;
    }
    if (c <= 0) c = choose_window_fixed_base(t->curve, n_hint ? n_hint : t->n, batch_hint ? batch_hint : 1);
    if (t->curve == kCurveBn254) precompute_impl<Bn254>(t, c, stream);
    else precompute_impl<Secp256k1>(t, c, stream);
    if (want_lut) {
        if (t->curve == kCurveBn254) lut_impl<Bn254>(t, stream);
        else lut_impl<Secp256k1>(t, stream);
    }
    return c;
}

// Total (scalar, bit) pairs up to which the one-launch bitwise tree sum beats the pipeline (latency of ~15
// dependent launches against n*bits/2 mixed additions of plain work).
static uint64_t small_bits_limit() {
    static const uint64_t v = [] {
        const char* e = getenv("PORLA_SMALL_BITS_LIMIT");
        return e ? (uint64_t)atoll(e) : (1ull << 18);
    }();
    return v;
}

MsmPlan msm_plan_table(const PointTable& t, uint32_t n, uint32_t nbatch, const MsmOptions& opt) {
    const bool fixed = t.fb_c > 0 && opt.shared_points && !opt.no_fixed_base &&
                       (opt.window_bits == 0 || opt.window_bits == t.fb_c);
    // PORLA_NO_SMALL=1 (or an explicit window size, PORLA_WINDOW_BITS included) keeps every call on the pipeline
    const char* ns = getenv("PORLA_NO_SMALL");
    const bool no_small = opt.no_small || (ns && ns[0] == '1') || getenv("PORLA_WINDOW_BITS");
    if (fixed) {
        const bool lut = t.d_lut && !no_small && nbatch <= 65535u && n <= t.n;
        return MsmPlan{t.fb_c, 1, lut ? kPlanLut : kPlanPipeline, 0};
    }
    if (opt.window_bits == 0 && !no_small && n > 0 && nbatch <= 65535u) {
        int bits = scalar_bits(t.curve);
        if (opt.max_scalar_bits > 0 && opt.max_scalar_bits < bits) bits = opt.max_scalar_bits;
        if ((uint64_t)n * nbatch * (uint64_t)bits <= small_bits_limit()) return MsmPlan{1, bits, kPlanBits, 0};
    }
    return msm_plan(t.curve, n, nbatch, opt.window_bits, opt.glv);
}

MsmPlan msm_plan(int curve, uint32_t n, uint32_t nbatch, int window_bits, int glv) {
    MsmPlan p;
    const WindowChoice ch = choose_window_ex(curve, n, nbatch, window_bits, glv);
    p.c = ch.c;
    p.glv = ch.glv;
    p.nwin = ((ch.glv ? Bn254::kGlvBits : scalar_bits(curve)) + 1 + p.c - 1) / p.c;
    p.mode = kPlanPipeline;
    return p;
}

size_t msm_bucket_bytes(const MsmPlan& plan) { return ((size_t)plan.nwin << (plan.c - 1)) * 128; }

// ---------------------------------------------------------------------------- host finaliser
template <class F64>
static void finalize_host_impl(const void* h_window_sums, int nparts, int nwin, int c, int out_fmt, uint8_t* out64) {
    static_assert(sizeof(XYZZ<F64>) == 128, "device and host XYZZ layouts must coincide");
    const XYZZ<F64>* ws = reinterpret_cast<const XYZZ<F64>*>(h_window_sums);
    XYZZ<F64> r = XYZZ<F64>::inf();
    for (int w = nwin - 1; w >= 0; w--) {
        if (!r.is_inf())
            for (int k = 0; k < c; k++) r = r.dbl();
        for (int part = 0; part < nparts; part++) {  // multi-GPU: one set of window sums per rank
            XYZZ<F64> s;
            memcpy(&s, ws + (size_t)part * nwin + w, sizeof(s));
            r.add(s);
        }
    }
    Affine<F64> a = r.to_affine();
    F64 xy[2] = {a.x.from_internal(), a.y.from_internal()};
    for (int k = 0; k < 2; k++) {
        if (out_fmt == 0) {  // big-endian
            for (int i = 0; i < 4; i++)
                for (int j = 0; j < 8; j++) out64[32 * k + 8 * (3 - i) + j] = (uint8_t)(xy[k].v[i] >> (8 * (7 - j)));
        } else {
            memcpy(out64 + 32 * k, xy[k].v, 32);
        }
    }
}

void finalize_host_parts(int curve, const void* h_window_sums, int nparts, int nwin, int c, int out_fmt, uint8_t* out64) {
    if (curve == kCurveBn254)
        finalize_host_impl<host::Fp64<host::Bn254Fq64Params>>(h_window_sums, nparts, nwin, c, out_fmt, out64);
    else
        finalize_host_impl<host::Fp64<host::SecpFq64Params>>(h_window_sums, nparts, nwin, c, out_fmt, out64);
}
void finalize_host(int curve, const void* h_window_sums, int nwin, int c, int out_fmt, uint8_t* out64) {
    finalize_host_parts(curve, h_window_sums, 1, nwin, c, out_fmt, out64);
}

// ---------------------------------------------------------------------------- dispatchers
void table_import_device(int curve, const uint8_t* d_bytes, int fmt, uint32_t n, PointTable* out, cudaStream_t stream) {
    device_init();
    DISPATCH(curve, import_impl, d_bytes, fmt, n, out, stream);
}

void table_import_host(int curve, const uint8_t* h_bytes, int fmt, uint32_t n, PointTable* out, cudaStream_t stream) {
    device_init();
    uint8_t* d_tmp = nullptr;
    PORLA_CUDA(cudaMalloc(&d_tmp, (size_t)(n ? n : 1) * 64));
    if (n) PORLA_CUDA(cudaMemcpyAsync(d_tmp, h_bytes, (size_t)n * 64, cudaMemcpyHostToDevice, stream));
    table_import_device(curve, d_tmp, fmt, n, out, stream);
    PORLA_CUDA(cudaFree(d_tmp));
}

void table_import_into(int curve, const uint8_t* d_bytes, int fmt, uint32_t n, void* d_points_out, uint8_t* d_flags_out,
                       PointTable* out, cudaStream_t stream, bool with_phi) {
    device_init();
    DISPATCH(curve, import_into_impl, d_bytes, fmt, n, d_points_out, d_flags_out, stream, with_phi);
    out->d_points = d_points_out;
    out->d_flags = d_flags_out;
    out->n = n;
    out->n_inf = 0;  // unknown (not counted on this path); the flags are always consulted
    out->curve = curve;
    out->phi_off = with_phi && curve == kCurveBn254 && Bn254::kGlv ? n : 0u;
    out->d_phi_x = out->phi_off ? static_cast<void*>(static_cast<uint8_t*>(d_points_out) + (size_t)n * 64) : nullptr;
}

void table_free(PointTable* t) {
    if (t->d_points) PORLA_CUDA(cudaFree(t->d_points));
    if (t->d_flags) PORLA_CUDA(cudaFree(t->d_flags));
    if (t->d_fb_points) PORLA_CUDA(cudaFree(t->d_fb_points));
    if (t->d_lut) PORLA_CUDA(cudaFree(t->d_lut));
    *t = PointTable{};
}

void msm_device(int curve, const PointTable& table, const uint8_t* d_scalars, uint32_t n, uint32_t nbatch,
                const MsmOptions& opt, uint8_t* d_out, void* d_out_xyzz, cudaStream_t stream) {
    device_init();
    if (nbatch == 0) return;
    DISPATCH(curve, msm_impl, table, d_scalars, n, nbatch, opt, d_out, d_out_xyzz, stream);
}

void msm_combine_device(int curve, const void* d_parts, uint32_t count, uint32_t nbatch, int out_fmt, uint8_t* d_out,
                        cudaStream_t stream) {
    device_init();
    if (nbatch == 0) return;
    DISPATCH(curve, combine_impl, d_parts, count, nbatch, out_fmt, d_out, stream);
}

void scalar_mul_device(int curve, const PointTable& table, const uint8_t* d_scalars, int scalar_be, uint32_t n,
                       void* d_out_affine, cudaStream_t stream) {
    device_init();
    if (!n) return;
    DISPATCH(curve, scalar_mul_impl, table, d_scalars, scalar_be, n, d_out_affine, stream);
}

void fixed_base_mul_device(int curve, const PointTable& table, const uint8_t* d_scalars, int scalar_be, uint32_t n, int out_fmt,
                           uint8_t* d_out, cudaStream_t stream) {
    device_init();
    if (table.n != 1 || !table.d_lut || table.curve != curve) {
        fprintf(stderr, "[libmultiexp/porla_b200] FATAL: fixed_base_mul_device needs a length-1 table of this curve with a look-up table\n");
        abort();
    }
    if (!n) return;
    DISPATCH(curve, fixed_base_mul_impl, table, d_scalars, scalar_be, n, out_fmt, d_out, stream);
}

void butterfly_stage_device(PointTable* t, uint32_t m, const uint8_t* d_twiddles, int scalar_be, cudaStream_t stream) {
    device_init();
    if (t->d_fb_points) {   // the expansion describes the old points
        PORLA_CUDA(cudaStreamSynchronize(stream));
        PORLA_CUDA(cudaFree(t->d_fb_points));
        if (t->d_lut) PORLA_CUDA(cudaFree(t->d_lut));
        t->d_fb_points = t->d_lut = nullptr;
        t->fb_c = t->fb_nwin = 0;
        t->fb_n = 0;
    }
    DISPATCH(t->curve, butterfly_impl, t, m, d_twiddles, scalar_be, stream);
}

void align_scalars_device(int curve, uint32_t* d_data, uint32_t total, uint8_t* d_scalars_be, cudaStream_t stream) {
    device_init();
    DISPATCH(curve, align_scalars_impl, d_data, total, d_scalars_be, stream);   // KZG mode: BN254 order, IPA mode: secp256k1's
}

void audit_aggregate_device(int curve, const uint32_t* d_coefs, const uint32_t* d_blocks, uint32_t n, uint32_t chunks,
                            uint8_t* d_b_mod_be, uint8_t* d_c_be, cudaStream_t stream) {
    device_init();
    DISPATCH(curve, audit_aggregate_impl, d_coefs, d_blocks, n, chunks, d_b_mod_be, d_c_be, stream);
}

void data_butterfly_launch(uint32_t*, uint32_t, uint32_t, uint32_t, const uint8_t*, const uint32_t*, const uint32_t*, cudaStream_t);

void data_butterfly_stage_device(uint32_t* d_blocks, uint32_t n_blocks, uint32_t chunks, uint32_t m, const uint8_t* d_twiddles,
                                 const uint8_t* lcm_le64, cudaStream_t stream) {
    device_init();
    uint32_t lcm[16];
    memcpy(lcm, lcm_le64, 64);
    // mu = floor(2^1022 / lcm) by restoring division (once per call, 1023 steps on 16 limbs)
    uint32_t mu[32] = {0}, rem[17] = {0};
    for (int bit = 1022; bit >= 0; bit--) {
        for (int i = 16; i > 0; i--) rem[i] = (rem[i] << 1) | (rem[i - 1] >> 31);   // rem = 2 rem + (bit of 2^1022)
        rem[0] = (rem[0] << 1) | (bit == 1022 ? 1u : 0u);
        uint32_t d[17];
        uint64_t borrow = 0;
        for (int i = 0; i < 17; i++) {
            uint64_t v = (uint64_t)rem[i] - (i < 16 ? lcm[i] : 0u) - borrow;
            d[i] = (uint32_t)v;
            borrow = (v >> 63) & 1;
        }
        if (!borrow) {
            memcpy(rem, d, sizeof(d));
            mu[bit >> 5] |= 1u << (bit & 31);
        }
    }
    for (int i = 17; i < 32; i++)
        if (mu[i]) {
            fprintf(stderr, "[libmultiexp/porla_b200] FATAL: data FFT modulus below 2^479\n");
            abort();
        }
    data_butterfly_launch(d_blocks, n_blocks, chunks, m, d_twiddles, lcm, mu, stream);
}

void export_points_device(int curve, const void* d_affine, uint32_t n, int fmt, uint8_t* d_out, cudaStream_t stream) {
    device_init();
    if (!n) return;
    DISPATCH(curve, export_impl, d_affine, n, fmt, d_out, stream);
}

void field_mul_device(int curve, const void* d_a, const void* d_b, uint32_t n, int op, void* d_out, cudaStream_t stream) {
    device_init();
    if (!n) return;
    DISPATCH(curve, field_mul_impl, d_a, d_b, n, op, d_out, stream);
}

}  // namespace porla
