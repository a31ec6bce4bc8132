// extern "C" surface of libmultiexp.so: the 14 cgo symbols of
// /root/reference/porla/Utils/libmultiexp.h:71-84 (Go bodies: /root/reference/porla/main.go) and the
// new batched / device-resident entry points declared in include/porla_multiexp.h.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <shared_mutex>
#include <thread>
#include <random>
#include <vector>

#include "../../include/porla_multiexp.h"
#include "bn254_pairing.hpp"
#include "host_bn254.hpp"
#include "msm.h"
#include "multi.h"
#include "staging.h"

using namespace porla;
using namespace porla::host;

namespace {

// ---------------------------------------------------------------------------- process state
// Mirrors the Go globals of main.go:18-29.
struct KzgState {
    Fr tau = Fr::zero(), alpha = Fr::zero();
    int64_t n_samples = 0;
    std::vector<G1A> srs_g1;        // host copy (internal form)
    G2A g2[2];                      // [1]G2, [tau]G2
    G2Lines g2_lines[2];            // their Miller-loop lines, precomputed once per SRS (verify_proof)
    bool have_g2 = false;
    G1A h_mac = G1A::inf();
    PointTable srs_table;           // resident in HBM
    bool have_table = false;
    bool lut_tried = false;         // the wide-window look-up table of a large batch is attempted once per upload
    uint64_t gen = 1;               // bumped (under g_srs_mu) whenever init_key / init_SRS* change tau, alpha, the SRS or h_MAC
};
KzgState g_kzg;

// Device state of the client's batched symbols (compute_digest_batch, compute_digest_complement_batch): length-1 tables
// of the digest base (the SRS's first point, [1]G1) and of h_MAC with their look-up tables, and the powers alpha tau^i in
// HBM.  Guarded by g_srs_mu like the SRS table; each part is rebuilt once its `*_gen` differs from g_kzg.gen.
struct ClientBase {
    porla_table t;
    uint64_t gen = 0;               // 0: never built
    bool wide_tried = false;        // the wide-window look-up table of a large batch is attempted once per build
};
struct ClientState {
    ClientBase digest, hmac;
    void* d_powers = nullptr;       // n_samples elements of Fr, Montgomery form
    uint64_t powers_gen = 0;
};
ClientState g_client;
}  // namespace

namespace {

// window_bits argument of the device entry points: a plain window size, or a plan code of porla_msm_plan
void decode_plan(int code, MsmOptions* opt) {
    opt->window_bits = PORLA_PLAN_WINDOW(code);
    opt->glv = (code & PORLA_PLAN_GLV_ON) ? 1 : (code & PORLA_PLAN_GLV_OFF) ? 0 : -1;
}

[[noreturn]] void die(const char* msg) {
    fprintf(stderr, "[libmultiexp/porla_b200] FATAL: %s\n", msg);
    abort();
}

// The engine indexes terms with 32 bits: refuse larger shapes at the boundary instead of letting the casts wrap.
void check_shape(int64_t n, int64_t nbatch, const char* what) {
    if (n < 0 || nbatch < 0 || n >= ((int64_t)1 << 31) || nbatch >= ((int64_t)1 << 31) ||
        (nbatch > 0 && n > (((int64_t)1 << 31) - 1) / nbatch)) {
        fprintf(stderr, "[libmultiexp/porla_b200] FATAL: %s: n = %lld, nbatch = %lld outside the supported range (n * nbatch < 2^31)\n",
                what, (long long)n, (long long)nbatch);
        abort();
    }
}

// Go's copy(dst, src): min(len(dst), len(src)) bytes
void go_copy(GoSlice* dst, const uint8_t* src, size_t n) {
    size_t k = (size_t)dst->len < n ? (size_t)dst->len : n;
    memcpy(dst->data, src, k);
}

std::vector<Fr> read_poly(const GoSlice* data_in, int64_t n) {
    if (data_in->len < n * 32) die("data_in shorter than n_samples*32 bytes (Go would panic: slice bounds out of range)");
    std::vector<Fr> f((size_t)n);
    const uint8_t* b = (const uint8_t*)data_in->data;
    for (int64_t i = 0; i < n; i++) f[(size_t)i] = elem_from_be<Fr>(b + 32 * i, 32);
    return f;
}

// Bit length of the largest scalar in a host buffer, or 0 when some scalar may need reduction (or, on
// secp256k1, the n - s recoding): lets small MSMs with short scalars (Porla's 31-bit audit coefficients,
// utils.h:271-275) run with one window per actual bit.
int host_max_scalar_bits(int curve, const uint8_t* scalars, size_t count, int big_endian) {
    int top_byte = -1;   // index (0 = least significant) of the highest non-zero byte over all scalars
    uint8_t top_val = 0;
    for (size_t i = 0; i < count; i++) {
        const uint8_t* s = scalars + 32 * i;
        for (int k = 31; k > top_byte; k--) {
            uint8_t v = big_endian ? s[31 - k] : s[k];
            if (v) {
                top_byte = k;
                top_val = 0;
                break;
            }
        }
        if (top_byte >= 0) {
            uint8_t v = big_endian ? s[31 - top_byte] : s[top_byte];
            if (v > top_val) top_val = v;
        }
    }
    if (top_byte < 0) return 1;
    int bits = 8 * top_byte;
    while (top_val) {
        bits++;
        top_val >>= 1;
    }
    const int limit = curve == kCurveBn254 ? 253 : 254;   // below 2^253 < r (BN254), below 2^254 < n/2 (secp256k1)
    return bits <= limit ? bits : 0;
}

// Host-buffer MSM core.  Scalars/points are copied to the device, points imported (the import
// kernel also decodes gnark's compressed-flag encodings), nbatch MSMs run, results copied back.
void msm_host_core(int curve, const uint8_t* scalars, const uint8_t* points, int64_t n, int64_t nbatch,
                   int scalar_fmt, int point_fmt, uint8_t* out) {
    if (nbatch <= 0) return;
    if (n <= 0) {
        memset(out, 0, (size_t)nbatch * 64);
        return;
    }
    check_shape(n, nbatch, "host-buffer MSM");
    device_init();
    if (nbatch == 1) {
        // a large call is partitioned by point range over the GPUs of the box, inside the call, as the reference
        // partitions it over 8 host threads (Client.hpp:747-787)
        const int ndev = fanout_devices(n);
        if (ndev > 1) {
            msm_host_fanout(curve, scalars, points, n, scalar_fmt, point_fmt, ndev, out);
            return;
        }
    }
    StagedCall call(n, nbatch);
    if (nbatch == 1 && n >= (1 << 19) && !getenv("PORLA_NO_SPLIT")) {
        // streamed: the terms cross PCIe in parts that are accumulated into one bucket set as they arrive (multi.cu)
        const MsmPlan plan = msm_plan(curve, (uint32_t)n, 1, 0);
        std::vector<uint8_t> ws((size_t)plan.nwin * 128);
        msm_host_pipelined(call.staging(), curve, scalars, points, n, scalar_fmt, point_fmt, plan, ws.data());
        finalize_host(curve, ws.data(), plan.nwin, plan.c, point_fmt, out);
        return;
    }
    const size_t total = (size_t)n * (size_t)nbatch;
    // staging layout: scalars | raw points | imported table + endomorphism image | infinity flags | result
    const size_t sc_bytes = total * 32, pt_bytes = total * 64;
    const size_t sc_off = call.add(sc_bytes), pt_off = call.add(pt_bytes), tab_off = call.add(2 * pt_bytes), fl_off = call.add(total);
    call.add_result(curve, n, nbatch);
    uint8_t* d = call.dev();
    cudaStream_t st = call.stream();
    h2d_copy(d + sc_off, scalars, sc_bytes, st);
    h2d_copy(d + pt_off, points, pt_bytes, st);
    MsmOptions opt = call.msm_options(scalar_fmt, point_fmt, 0);
    if (total <= 4096) opt.max_scalar_bits = host_max_scalar_bits(curve, scalars, total, opt.scalar_be);
    PointTable tab;
    tab.curve = curve;
    // the one-launch tree sum does not use the endomorphism image: skip that launch for Porla-sized calls
    const bool bits_plan = msm_plan_table(tab, (uint32_t)n, (uint32_t)nbatch, opt).mode == kPlanBits;
    table_import_into(curve, d + pt_off, point_fmt, (uint32_t)total, d + tab_off, d + fl_off, &tab, st, !bits_plan);
    call.fetch(curve, tab, d + sc_off, n, nbatch, opt, out);
}

void upload_srs_locked();

// g_kzg.srs_table is read by every commitment (also by the small calls that take no other lock) and rebuilt in two
// places: the first upload and the one-time wide-window look-up table of a large batch.  Readers hold g_srs_mu shared
// for the whole call, the two writers hold it exclusively (so no kernel of a reader can still be using pointers that
// table_precompute frees: every reader synchronises its stream before it drops the lock).
std::shared_mutex g_srs_mu;

// Shared lock on the SRS table with the table present and at least `n` bases long; `batch_terms` = n * nbatch of the
// call (a large batch over a mid-sized SRS, BASELINE config 3, is worth the one-time wide-window look-up table).
std::shared_lock<std::shared_mutex> srs_reader(int64_t n, uint64_t batch_terms, int64_t nbatch) {
    auto want_lut = [&] {   // read under g_srs_mu
        return batch_terms >= (1ull << 22) && g_kzg.srs_table.n > 2048 && g_kzg.srs_table.n <= 8192 && !g_kzg.srs_table.d_lut &&
               !g_kzg.lut_tried && !getenv("PORLA_NO_LUT");
    };
    for (;;) {
        {
            std::shared_lock<std::shared_mutex> rd(g_srs_mu);
            if (g_kzg.have_table && !want_lut()) {
                if (n > (int64_t)g_kzg.srs_table.n) die("polynomial longer than the SRS");
                return rd;
            }
        }
        std::unique_lock<std::shared_mutex> wr(g_srs_mu);
        if (!g_kzg.have_table) {
            if (g_kzg.srs_g1.empty()) die("SRS not initialised (call init_SRS or init_SRS_from_data first)");
            upload_srs_locked();
        }
        if (want_lut()) {
            StagedCall call;
            table_precompute(&g_kzg.srs_table, 0, (uint32_t)n, (uint32_t)nbatch, call.stream());
            PORLA_CUDA(cudaStreamSynchronize(call.stream()));
            g_kzg.lut_tried = true;
        }
    }
}

// nbatch commitments over the resident SRS
void srs_commit_core(const uint8_t* coeffs_be, int64_t n, int64_t nbatch, uint8_t* out) {
    check_shape(n, nbatch, "commitment over the SRS");
    device_init();
    std::shared_lock<std::shared_mutex> srs = srs_reader(n, (uint64_t)n * (uint64_t)nbatch, nbatch);
    StagedCall call(n, nbatch);
    const size_t sc_bytes = (size_t)n * nbatch * 32;
    call.add(sc_bytes);
    call.add_result(kCurveBn254, n, nbatch);
    uint8_t* d = call.dev();
    h2d_copy(d, coeffs_be, sc_bytes, call.stream());
    call.fetch(kCurveBn254, g_kzg.srs_table, d, n, nbatch, call.msm_options(PORLA_SCALAR_BE32, PORLA_POINT_BE64, 1), out);
}

// SRS bases go to HBM once, at init when a device is present (otherwise on the first commit,
// which aborts loudly if there is still no GPU).
// Caller holds g_srs_mu exclusively.
void upload_srs_locked() {
    device_init();
    StagedCall call;
    if (g_kzg.srs_table.d_points) table_free(&g_kzg.srs_table);
    std::vector<uint8_t> bytes(g_kzg.srs_g1.size() * 64);
    for (size_t i = 0; i < g_kzg.srs_g1.size(); i++) g1_marshal(g_kzg.srs_g1[i], bytes.data() + 64 * i);
    table_import_host(kCurveBn254, bytes.data(), PORLA_POINT_BE64, (uint32_t)g_kzg.srs_g1.size(), &g_kzg.srs_table,
                      call.stream());
    // the SRS is a fixed base: expand it once so that commitments need no per-window reduction
    if (!getenv("PORLA_NO_FIXED_BASE")) {
        table_precompute(&g_kzg.srs_table, 0, (uint32_t)g_kzg.srs_g1.size(), 1, call.stream());
        PORLA_CUDA(cudaStreamSynchronize(call.stream()));
    }
    g_kzg.have_table = true;
    g_kzg.lut_tried = false;
}

void upload_srs() {
    std::unique_lock<std::shared_mutex> wr(g_srs_mu);
    upload_srs_locked();
}

void kzg_state_changed() {
    std::unique_lock<std::shared_mutex> wr(g_srs_mu);
    g_kzg.gen++;
}

// A batch of at least this many scalars over one base is worth the wide-window look-up table (table_precompute's
// n_hint * batch_hint threshold with n_hint = 1: c = 16, 16 windows, 32 MiB).
constexpr int64_t kWideBatch = (int64_t)1 << 22;

bool client_base_fresh(const ClientBase& b, int64_t batch) {
    return b.gen == g_kzg.gen && !(batch >= kWideBatch && !b.wide_tried && !getenv("PORLA_NO_LUT"));
}

// Caller holds g_srs_mu exclusively.  The base goes through the same import and precompute as any resident table:
// table_precompute with window_bits = 0 gives a length-1 table the c = 8 look-up table, or the wide one for a large batch.
void client_base_build(ClientBase* b, const G1A& base, int64_t batch) {
    device_init();
    StagedCall call;
    if (b->t.t.d_points) table_free(&b->t.t);   // no reader left: each synchronised its stream before dropping g_srs_mu
    uint8_t bytes[64];
    g1_marshal(base, bytes);
    table_import_host(kCurveBn254, bytes, PORLA_POINT_BE64, 1, &b->t.t, call.stream());
    table_precompute(&b->t.t, 0, 1, (uint32_t)(batch > 0 ? batch : 1), call.stream());
    PORLA_CUDA(cudaStreamSynchronize(call.stream()));
    b->gen = g_kzg.gen;
    b->wide_tried = batch >= kWideBatch;
}

// Caller holds g_srs_mu exclusively.
void client_powers_build() {
    device_init();
    if (g_client.d_powers) PORLA_CUDA(cudaFree(g_client.d_powers));
    g_client.d_powers = nullptr;
    const int64_t n = g_kzg.n_samples;
    if (n > 0) {
        std::vector<Fr> p((size_t)n);
        Fr acc = g_kzg.alpha;
        for (int64_t i = 0; i < n; i++) {
            p[(size_t)i] = acc;
            acc = acc * g_kzg.tau;
        }
        PORLA_CUDA(cudaMalloc(&g_client.d_powers, (size_t)n * sizeof(Fr)));
        PORLA_CUDA(cudaMemcpy(g_client.d_powers, p.data(), (size_t)n * sizeof(Fr), cudaMemcpyHostToDevice));
    }
    g_client.powers_gen = g_kzg.gen;
}

// Shared lock on the client state with the digest table and powers (digest) or the h_MAC table current for the calling
// state of init_key / init_SRS*, rebuilding what is stale under the exclusive lock first.
std::shared_lock<std::shared_mutex> client_reader(bool digest, int64_t batch) {
    auto fresh = [&] {
        return digest ? client_base_fresh(g_client.digest, batch) && g_client.powers_gen == g_kzg.gen
                      : client_base_fresh(g_client.hmac, batch);
    };
    for (;;) {
        {
            std::shared_lock<std::shared_mutex> rd(g_srs_mu);
            if (fresh()) return rd;
        }
        std::unique_lock<std::shared_mutex> wr(g_srs_mu);
        if (digest) {
            if (!client_base_fresh(g_client.digest, batch))
                client_base_build(&g_client.digest, g_kzg.srs_g1.empty() ? g1_generator() : g_kzg.srs_g1[0], batch);
            if (g_client.powers_gen != g_kzg.gen) client_powers_build();
        } else if (!client_base_fresh(g_client.hmac, batch)) {
            client_base_build(&g_client.hmac, g_kzg.h_mac, batch);
        }
    }
}

// `batch` fixed-base products over a length-1 table (d_scalars already queued on the call's stream); returns the call's
// pinned buffer holding the batch x 64 result bytes (out_fmt).
const uint8_t* fixed_base_products(StagedCall& call, const porla_table* base, const uint8_t* d_scalars, int scalar_fmt,
                                   int64_t batch, int out_fmt, uint8_t* d_out) {
    porla_scalar_mul_batch_device(base, d_scalars, batch, scalar_fmt, out_fmt, d_out, call.stream());
    uint8_t* h = call.pinned((size_t)batch * 64);
    PORLA_CUDA(cudaMemcpyAsync(h, d_out, (size_t)batch * 64, cudaMemcpyDeviceToHost, call.stream()));
    PORLA_CUDA(cudaStreamSynchronize(call.stream()));
    return h;
}

}  // namespace

namespace porla {

PointTable table_window(const PointTable& t, int64_t first, int64_t n) {
    PointTable view = t;
    view.d_points = (uint8_t*)t.d_points + (size_t)first * 64;
    view.d_flags = t.d_flags ? t.d_flags + first : nullptr;
    view.n = (uint32_t)n;
    if (t.d_phi_x) {                           // image of entry first + i: same index arithmetic on the beta*x array
        view.d_phi_x = (uint8_t*)t.d_phi_x + (size_t)first * 32;
        view.phi_off = (uint32_t)n;
    }
    if (t.fb_c > 0) {                          // the expansion's rows keep their stride; start them at `first`
        view.d_fb_points = (uint8_t*)t.d_fb_points + (size_t)first * 64;
        if (t.d_lut) view.d_lut = (uint8_t*)t.d_lut + ((((size_t)first * t.fb_nwin) << (t.fb_c - 1)) * 64);
    }
    return view;
}

void align_mac_core(int curve, const PointTable& gens, void* data, int64_t n, int64_t batch, int out_fmt, uint8_t* out) {
    if (batch == 0) return;
    device_init();
    StagedCall call(n, batch);
    const size_t total = (size_t)batch * n;
    call.add(total * 64);
    const size_t sc_off = call.add(total * 32);
    call.add_result(curve, n, batch);
    uint8_t* d = call.dev();
    cudaStream_t st = call.stream();
    h2d_copy(d, data, total * 64, st);
    align_scalars_device(curve, reinterpret_cast<uint32_t*>(d), (uint32_t)total, d + sc_off, st);
    PORLA_CUDA(cudaMemcpyAsync(data, d, total * 64, cudaMemcpyDeviceToHost, st));   // A[i] <- A[i] % PRIME_MODULUS
    call.fetch(curve, gens, d + sc_off, n, batch, call.msm_options(PORLA_SCALAR_BE32, out_fmt, 1), out);
}

void audit_aggregate_core(int curve, const PointTable& gens, const void* coefs, const void* blocks, int64_t n, int64_t chunks,
                          int out_fmt, uint8_t* b_mod_be, uint8_t* out64) {
    device_init();
    // the blocks are the call's volume: a slot is leased when they are no more than a small MSM's terms
    StagedCall call((n > 0 ? n : 1) * chunks, 1);
    const size_t blk_bytes = (size_t)n * chunks * 64;
    call.add(blk_bytes);
    const size_t cf_off = call.add((size_t)n * 4 + 4), b_off = call.add((size_t)chunks * 32), c_off = call.add((size_t)chunks * 32);
    call.add_result(curve, chunks, 1);
    uint8_t* d = call.dev();
    cudaStream_t st = call.stream();
    if (n) {
        h2d_copy(d, blocks, blk_bytes, st);
        PORLA_CUDA(cudaMemcpyAsync(d + cf_off, coefs, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    }
    audit_aggregate_device(curve, reinterpret_cast<const uint32_t*>(d + cf_off), reinterpret_cast<const uint32_t*>(d), (uint32_t)n,
                           (uint32_t)chunks, d + b_off, d + c_off, st);
    PORLA_CUDA(cudaMemcpyAsync(b_mod_be, d + b_off, (size_t)chunks * 32, cudaMemcpyDeviceToHost, st));
    call.fetch(curve, gens, d + c_off, chunks, 1, call.msm_options(PORLA_SCALAR_BE32, out_fmt, 1), out64);
}

void msm_host_jacobian_secp256k1(const uint32_t* xyz, const uint8_t* inf, const void* scalars, int64_t n, int64_t nbatch,
                                 uint8_t* out) {
    check_shape(n, nbatch, "secp256k1 Jacobian MSM");
    device_init();
    StagedCall call(n, nbatch);
    const size_t total = (size_t)n * nbatch;
    // staging layout: scalars | X, Y, Z | infinity flags in | affine table | its flags | result
    call.add(total * 32);
    const size_t xyz_off = call.add(total * 96), inf_off = call.add(total), tab_off = call.add(total * 64), fl_off = call.add(total);
    call.add_result(kCurveSecp256k1, n, nbatch);
    uint8_t* d = call.dev();
    cudaStream_t st = call.stream();
    h2d_copy(d, scalars, total * 32, st);
    h2d_copy(d + xyz_off, xyz, total * 96, st);
    h2d_copy(d + inf_off, inf, total, st);
    MsmOptions opt = call.msm_options(PORLA_SCALAR_LE32, PORLA_POINT_LE64, 0);
    if (total <= 4096) opt.max_scalar_bits = host_max_scalar_bits(kCurveSecp256k1, (const uint8_t*)scalars, total, 0);
    PointTable tab;
    table_import_jacobian_secp256k1(reinterpret_cast<const uint32_t*>(d + xyz_off), d + inf_off, (uint32_t)total, d + tab_off,
                                    d + fl_off, &tab, st);
    call.fetch(kCurveSecp256k1, tab, d, n, nbatch, opt, out);
}

const uint8_t* fixed_base_mul_core(StagedCall& call, const porla_table* base, const void* scalars, int64_t n, int scalar_fmt,
                                   int out_fmt) {
    const size_t sc_bytes = (size_t)n * 32;
    call.add(sc_bytes);
    const size_t out_off = call.add((size_t)n * 64);
    uint8_t* d = call.dev();
    h2d_copy(d, scalars, sc_bytes, call.stream());
    return fixed_base_products(call, base, d, scalar_fmt, n, out_fmt, d + out_off);
}

}  // namespace porla

extern "C" {

// ============================================================================ legacy cgo ABI
void init_key(GoSlice* tau_key_in, GoSlice* alpha_key_in) {
    g_kzg.tau = elem_from_be<Fr>((const uint8_t*)tau_key_in->data, (size_t)tau_key_in->len);
    g_kzg.alpha = elem_from_be<Fr>((const uint8_t*)alpha_key_in->data, (size_t)alpha_key_in->len);
    kzg_state_changed();
}

void init_SRS(GoInt SRS_size, GoSlice* out, GoInt64* out_len) {
    if (SRS_size <= 0) die("init_SRS: SRS_size must be positive");
    g_kzg.n_samples = SRS_size;
    // kzg.NewSRS: G1[i] = [tau^i]G1, G2 = {G2, [tau]G2}
    g_kzg.srs_g1.resize((size_t)SRS_size);
    G1A g = g1_generator();
    Fr t = Fr::one();
    for (GoInt i = 0; i < SRS_size; i++) {
        g_kzg.srs_g1[(size_t)i] = g1_mul(g, t);
        t = t * g_kzg.tau;
    }
    g_kzg.g2[0] = g2_generator();
    g_kzg.g2[1] = g2_mul(g_kzg.g2[0], g_kzg.tau);
    for (int i = 0; i < 2; i++) g_kzg.g2_lines[i] = g2_precompute_lines(g_kzg.g2[i]);
    g_kzg.have_g2 = true;
    // SRS.WriteTo: compressed encoder over &G2[0], &G2[1], G1 (uint32 BE length prefix)
    std::vector<uint8_t> blob(128 + 4 + (size_t)SRS_size * 32);
    g2_compress(g_kzg.g2[0], blob.data());
    g2_compress(g_kzg.g2[1], blob.data() + 64);
    uint32_t cnt = (uint32_t)SRS_size;
    blob[128] = (uint8_t)(cnt >> 24);
    blob[129] = (uint8_t)(cnt >> 16);
    blob[130] = (uint8_t)(cnt >> 8);
    blob[131] = (uint8_t)cnt;
    for (GoInt i = 0; i < SRS_size; i++) g1_compress(g_kzg.srs_g1[(size_t)i], blob.data() + 132 + 32 * i);
    *out_len = (GoInt64)blob.size();
    go_copy(out, blob.data(), blob.size());
    // h_MAC = [rho]G1, rho random (main.go:52-59)
    std::random_device rd;
    uint8_t rb[32];
    for (int i = 0; i < 32; i += 4) {
        uint32_t v = rd();
        memcpy(rb + i, &v, 4);
    }
    g_kzg.h_mac = g1_mul(g, elem_from_be<Fr>(rb, 32));
    g_kzg.have_table = false;
    kzg_state_changed();
    if (device_available()) upload_srs();
}

void init_SRS_from_data(GoInt SRS_size, GoSlice* in) {
    if (SRS_size <= 0) die("init_SRS_from_data: SRS_size must be positive");
    const uint8_t* b = (const uint8_t*)in->data;
    if (in->len < 132) die("init_SRS_from_data: blob too short");
    g_kzg.n_samples = SRS_size;
    if (!g2_decompress(b, &g_kzg.g2[0]) || !g2_decompress(b + 64, &g_kzg.g2[1])) die("init_SRS_from_data: bad G2 point");
    for (int i = 0; i < 2; i++) g_kzg.g2_lines[i] = g2_precompute_lines(g_kzg.g2[i]);
    g_kzg.have_g2 = true;
    uint32_t cnt = ((uint32_t)b[128] << 24) | ((uint32_t)b[129] << 16) | ((uint32_t)b[130] << 8) | b[131];
    if ((GoInt)in->len < 132 + (GoInt)cnt * 32) die("init_SRS_from_data: blob truncated");
    g_kzg.srs_g1.resize(cnt);
    for (uint32_t i = 0; i < cnt; i++)
        if (!g1_unmarshal(b + 132 + 32 * (size_t)i, 32, &g_kzg.srs_g1[i])) die("init_SRS_from_data: bad G1 point");
    g_kzg.have_table = false;
    kzg_state_changed();
    if (device_available()) upload_srs();
}

void compute_digest(GoSlice* data_in, GoSlice* data_out) {
    std::vector<Fr> f = read_poly(data_in, g_kzg.n_samples);
    Fr fx = poly_eval(f, g_kzg.tau) * g_kzg.alpha;
    G1A base = g_kzg.srs_g1.empty() ? g1_generator() : g_kzg.srs_g1[0];
    uint8_t buf[64];
    g1_marshal(g1_mul(base, fx), buf);
    go_copy(data_out, buf, 64);
}

void compute_digest_complement(GoSlice* data_in, GoSlice* data_out) {
    Fr s = elem_from_be<Fr>((const uint8_t*)data_in->data, (size_t)data_in->len);
    uint8_t buf[64];
    g1_marshal(g1_mul(g_kzg.h_mac, s), buf);
    go_copy(data_out, buf, 64);
}

void compute_digest_from_srs(GoSlice* data_in, GoSlice* data_out) {
    if (data_in->len < g_kzg.n_samples * 32) die("compute_digest_from_srs: data_in too short");
    uint8_t buf[64];
    srs_commit_core((const uint8_t*)data_in->data, g_kzg.n_samples, 1, buf);
    go_copy(data_out, buf, 64);
}

void compute_multi_exp(GoSlice* scalars, GoSlice* points, GoInt length, GoSlice* result_out) {
    if (length < 0 || scalars->len < length * 32 || points->len < length * 64)
        die("compute_multi_exp: slices shorter than length (Go would panic: slice bounds out of range)");
    uint8_t buf[64];
    msm_host_core(kCurveBn254, (const uint8_t*)scalars->data, (const uint8_t*)points->data, length, 1,
                  PORLA_SCALAR_BE32, PORLA_POINT_BE64, buf);
    go_copy(result_out, buf, 64);
}

GoUint8 compare_commitment(GoSlice* commitment_a, GoSlice* commitment_b) {
    G1A a = G1A::inf(), b = G1A::inf();
    g1_unmarshal((const uint8_t*)commitment_a->data, (size_t)commitment_a->len, &a);
    g1_unmarshal((const uint8_t*)commitment_b->data, (size_t)commitment_b->len, &b);
    if (!(a.x == b.x && a.y == b.y)) {
        printf("error KZG commitment\n");
        return 0;
    }
    return 1;
}

void create_proof(GoUint64 random_point, GoSlice* data_in, GoSlice* commitment_out, GoSlice* proof_H,
                  GoSlice* proof_point, GoSlice* proof_claim) {
    const int64_t n = g_kzg.n_samples;
    std::vector<Fr> f = read_poly(data_in, n);
    Fr z = elem_from_u64<Fr>(random_point);
    Fr y = poly_eval(f, z);
    std::vector<Fr> h = poly_quotient(f, z);
    // both commitments in one launch sequence: MSM 0 = f (n terms), MSM 1 = h padded with a zero
    std::vector<uint8_t> coeffs((size_t)n * 64, 0);
    memcpy(coeffs.data(), data_in->data, (size_t)n * 32);
    for (size_t i = 0; i < h.size(); i++) elem_to_be(h[i], coeffs.data() + (size_t)n * 32 + 32 * i);
    uint8_t res[128];
    srs_commit_core(coeffs.data(), n, 2, res);
    go_copy(commitment_out, res, 64);
    go_copy(proof_H, res + 64, 64);
    uint8_t buf[32];
    elem_to_be(z, buf);
    go_copy(proof_point, buf, 32);
    elem_to_be(y, buf);
    go_copy(proof_claim, buf, 32);
}

GoUint8 verify_proof(GoSlice* commitment_in, GoSlice* proof_H, GoSlice* proof_point, GoSlice* proof_claim) {
    G1A c = G1A::inf(), hq = G1A::inf();
    g1_unmarshal((const uint8_t*)commitment_in->data, (size_t)commitment_in->len, &c);
    g1_unmarshal((const uint8_t*)proof_H->data, (size_t)proof_H->len, &hq);
    Fr z = elem_from_be<Fr>((const uint8_t*)proof_point->data, (size_t)proof_point->len);
    Fr y = elem_from_be<Fr>((const uint8_t*)proof_claim->data, (size_t)proof_claim->len);
    if (!g_kzg.have_g2) die("verify_proof: SRS not initialised");
    // kzg.Verify checks e(C - [y]G1, G2) * e(-H, [tau]G2 - [z]G2) == 1.  By bilinearity
    // e(-H, -[z]G2) = e([z]H, G2), so the same predicate is e(C - [y]G1 + [z]H, G2) * e(-H, [tau]G2) == 1:
    // only G1 scalar multiplications, and both G2 arguments are the fixed SRS points.
    G1A yg = g1_mul(g_kzg.srs_g1.empty() ? g1_generator() : g_kzg.srs_g1[0], y);
    G1A lhs = g1_add(g1_add(c, yg.neg()), g1_mul(hq, z));
    G1A ps[2] = {lhs, hq.neg()};
    G2A qs[2] = {g_kzg.g2[0], g_kzg.g2[1]};
    const G2Lines* ls[2] = {&g_kzg.g2_lines[0], &g_kzg.g2_lines[1]};
    const bool fixed = ls[0]->valid && ls[1]->valid && !getenv("PORLA_PAIRING_GENERIC");
    if (!(fixed ? pairing_product_is_one_fixed(ps, ls, 2) : pairing_product_is_one(ps, qs, 2))) {
        printf("Verifying is wrong\n");
        return 0;
    }
    return 1;
}

void add_point(GoSlice* point_a, GoSlice* point_b) {
    G1A a = G1A::inf(), b = G1A::inf();
    g1_unmarshal((const uint8_t*)point_a->data, (size_t)point_a->len, &a);
    g1_unmarshal((const uint8_t*)point_b->data, (size_t)point_b->len, &b);
    uint8_t buf[64];
    g1_marshal(g1_add(a, b), buf);
    go_copy(point_a, buf, 64);
}

void mult_point(GoSlice* point_a, GoSlice* scalar) {
    G1A p = G1A::inf();
    g1_unmarshal((const uint8_t*)point_a->data, (size_t)point_a->len, &p);
    Fr s = elem_from_be<Fr>((const uint8_t*)scalar->data, (size_t)scalar->len);
    uint8_t buf[64];
    g1_marshal(g1_mul(p, s), buf);
    go_copy(point_a, buf, 64);
}

void neg_point(GoSlice* point) {
    G1A p = G1A::inf();
    g1_unmarshal((const uint8_t*)point->data, (size_t)point->len, &p);
    uint8_t buf[64];
    g1_marshal(p.neg(), buf);
    go_copy(point, buf, 64);
}

void set_inf_point(GoSlice* point) {
    uint8_t buf[64] = {0};
    go_copy(point, buf, 64);
}

// ============================================================================ new entry points
int porla_device_init(void) { return device_init(); }
uint64_t porla_launch_count(void) { return launches_issued(); }
void porla_stage_timing_enable(int on) { stage_timing_enable(on); }
int porla_stage_timing_read(float* ms_out) { return stage_timing_read(ms_out); }
int porla_choose_window(int curve, int64_t n, int64_t nbatch) { return choose_window(curve, (uint32_t)n, (uint32_t)nbatch); }

void compute_multi_exp_batch(GoSlice* scalars, GoSlice* points, GoInt length, GoInt batch, GoSlice* results_out) {
    if (length < 0 || batch < 0 || scalars->len < length * batch * 32 || points->len < length * batch * 64)
        die("compute_multi_exp_batch: slices shorter than batch*length");
    std::vector<uint8_t> buf((size_t)batch * 64);
    msm_host_core(kCurveBn254, (const uint8_t*)scalars->data, (const uint8_t*)points->data, length, batch,
                  PORLA_SCALAR_BE32, PORLA_POINT_BE64, buf.data());
    go_copy(results_out, buf.data(), buf.size());
}

void compute_digest_from_srs_batch(GoSlice* data_in, GoInt batch, GoSlice* data_out) {
    if (batch < 0 || data_in->len < g_kzg.n_samples * 32 * batch) die("compute_digest_from_srs_batch: data_in too short");
    std::vector<uint8_t> buf((size_t)batch * 64);
    if (batch) srs_commit_core((const uint8_t*)data_in->data, g_kzg.n_samples, batch, buf.data());
    go_copy(data_out, buf.data(), buf.size());
}

void compute_digest_batch(GoSlice* data_in, GoInt batch, GoSlice* data_out) {
    const int64_t n = g_kzg.n_samples;
    if (batch < 0 || data_in->len < n * 32 * batch) die("compute_digest_batch: data_in shorter than batch*n_samples*32 bytes");
    if (batch == 0) return;
    check_shape(n, batch, "compute_digest_batch");
    device_init();
    std::shared_lock<std::shared_mutex> rd = client_reader(true, batch);
    StagedCall call(n, batch);
    const size_t co_bytes = (size_t)n * batch * 32;
    call.add(co_bytes);
    const size_t sc_off = call.add((size_t)batch * 32), out_off = call.add((size_t)batch * 64);
    uint8_t* d = call.dev();
    if (co_bytes) h2d_copy(d, data_in->data, co_bytes, call.stream());
    // alpha * f(tau) per record on the device, then [.]G1 over the resident table of the digest base
    fr_poly_eval_device(d, g_client.d_powers, (uint32_t)n, (uint32_t)batch, d + sc_off, call.stream());
    const uint8_t* h = fixed_base_products(call, &g_client.digest.t, d + sc_off, PORLA_SCALAR_LE32, batch, PORLA_POINT_BE64, d + out_off);
    go_copy(data_out, h, (size_t)batch * 64);
}

void compute_digest_complement_batch(GoSlice* data_in, GoInt batch, GoSlice* data_out) {
    if (batch < 0 || data_in->len < batch * 32) die("compute_digest_complement_batch: data_in shorter than batch*32 bytes");
    if (batch == 0) return;
    check_shape(1, batch, "compute_digest_complement_batch");
    device_init();
    std::shared_lock<std::shared_mutex> rd = client_reader(false, batch);
    StagedCall call(1, batch);
    go_copy(data_out, fixed_base_mul_core(call, &g_client.hmac.t, data_in->data, batch, PORLA_SCALAR_BE32, PORLA_POINT_BE64),
            (size_t)batch * 64);
}

porla_table* porla_table_create(int curve, const void* points, int64_t n, int point_fmt, int on_device, void* cuda_stream) {
    check_shape(n, 1, "porla_table_create");
    device_init();
    porla_table* t = new porla_table();
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if (on_device) table_import_device(curve, (const uint8_t*)points, point_fmt, (uint32_t)n, &t->t, st);
    else table_import_host(curve, (const uint8_t*)points, point_fmt, (uint32_t)n, &t->t, st);
    return t;
}

porla_table* porla_table_create_multiples(int curve, const void* scalars, int64_t n, int scalar_fmt, int on_device,
                                          void* cuda_stream) {
    check_shape(n, 1, "porla_table_create_multiples");
    device_init();
    cudaStream_t st = (cudaStream_t)cuda_stream;
    // generator as a 1-entry table
    uint8_t gen[64] = {0};
    if (curve == kCurveBn254) {
        gen[31] = 1;
        gen[63] = 2;
    } else {
        static const uint8_t sg[64] = {
            0x79, 0xBE, 0x66, 0x7E, 0xF9, 0xDC, 0xBB, 0xAC, 0x55, 0xA0, 0x62, 0x95, 0xCE, 0x87, 0x0B, 0x07,
            0x02, 0x9B, 0xFC, 0xDB, 0x2D, 0xCE, 0x28, 0xD9, 0x59, 0xF2, 0x81, 0x5B, 0x16, 0xF8, 0x17, 0x98,
            0x48, 0x3A, 0xDA, 0x77, 0x26, 0xA3, 0xC4, 0x65, 0x5D, 0xA4, 0xFB, 0xFC, 0x0E, 0x11, 0x08, 0xA8,
            0xFD, 0x17, 0xB4, 0x48, 0xA6, 0x85, 0x54, 0x19, 0x9C, 0x47, 0xD0, 0x8F, 0xFB, 0x10, 0xD4, 0xB8};
        memcpy(gen, sg, 64);
    }
    PointTable g;
    table_import_host(curve, gen, PORLA_POINT_BE64, 1, &g, st);
    const uint8_t* d_sc = (const uint8_t*)scalars;
    uint8_t* d_tmp = nullptr;
    if (!on_device) {
        PORLA_CUDA(cudaMalloc(&d_tmp, (size_t)n * 32));
        PORLA_CUDA(cudaMemcpyAsync(d_tmp, scalars, (size_t)n * 32, cudaMemcpyHostToDevice, st));
        d_sc = d_tmp;
    }
    porla_table* t = new porla_table();
    void* d_aff = nullptr;
    PORLA_CUDA(cudaMalloc(&d_aff, (size_t)(n ? n : 1) * 64));
    scalar_mul_device(curve, g, d_sc, scalar_fmt == PORLA_SCALAR_BE32, (uint32_t)n, d_aff, st);
    // re-import through the external format so infinity flags are derived the same way
    uint8_t* d_ext = nullptr;
    PORLA_CUDA(cudaMalloc(&d_ext, (size_t)(n ? n : 1) * 64));
    export_points_device(curve, d_aff, (uint32_t)n, PORLA_POINT_LE64, d_ext, st);
    table_import_device(curve, d_ext, PORLA_POINT_LE64, (uint32_t)n, &t->t, st);
    PORLA_CUDA(cudaStreamSynchronize(st));
    PORLA_CUDA(cudaFree(d_ext));
    PORLA_CUDA(cudaFree(d_aff));
    if (d_tmp) PORLA_CUDA(cudaFree(d_tmp));
    table_free(&g);
    return t;
}

int porla_table_precompute(porla_table* t, int window_bits, int64_t n_hint, int64_t batch_hint, void* cuda_stream) {
    int c = table_precompute(&t->t, window_bits, (uint32_t)n_hint, (uint32_t)batch_hint, (cudaStream_t)cuda_stream);
    PORLA_CUDA(cudaStreamSynchronize((cudaStream_t)cuda_stream));
    return c;
}

int64_t porla_table_len(const porla_table* t) { return t->t.n; }
int64_t porla_table_num_infinity(const porla_table* t) { return t->t.n_inf; }

void porla_table_export(const porla_table* t, int point_fmt, void* out, int on_device, void* cuda_stream) {
    device_init();
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if (on_device) {
        export_points_device(t->t.curve, t->t.d_points, t->t.n, point_fmt, (uint8_t*)out, st);
        return;
    }
    uint8_t* d = nullptr;
    PORLA_CUDA(cudaMalloc(&d, (size_t)(t->t.n ? t->t.n : 1) * 64));
    export_points_device(t->t.curve, t->t.d_points, t->t.n, point_fmt, d, st);
    PORLA_CUDA(cudaMemcpyAsync(out, d, (size_t)t->t.n * 64, cudaMemcpyDeviceToHost, st));
    PORLA_CUDA(cudaStreamSynchronize(st));
    PORLA_CUDA(cudaFree(d));
}

void porla_table_destroy(porla_table* t) {
    if (!t) return;
    table_free(&t->t);
    delete t;
}

void porla_msm_device(const porla_table* t, const void* d_scalars, int64_t n, int64_t nbatch, int scalar_fmt,
                      int shared_points, int window_bits, int out_fmt, void* d_out, void* d_out_xyzz, void* cuda_stream) {
    check_shape(n, nbatch, "porla_msm_device");
    int64_t need = shared_points ? n : n * nbatch;
    if (need > (int64_t)t->t.n) die("porla_msm_device: table shorter than the MSM");
    MsmOptions opt;
    decode_plan(window_bits, &opt);
    opt.scalar_be = scalar_fmt == PORLA_SCALAR_BE32;
    opt.out_fmt = out_fmt;
    opt.shared_points = shared_points;
    msm_device(t->t.curve, t->t, (const uint8_t*)d_scalars, (uint32_t)n, (uint32_t)nbatch, opt, (uint8_t*)d_out, d_out_xyzz,
               (cudaStream_t)cuda_stream);
}

void porla_msm_resident(const porla_table* t, const void* d_scalars, int64_t n, int scalar_fmt, int window_bits, int out_fmt,
                        void* h_out64, void* cuda_stream) {
    if (n > (int64_t)t->t.n) die("porla_msm_resident: table shorter than the MSM");
    if (n <= 0) {
        memset(h_out64, 0, 64);
        return;
    }
    check_shape(n, 1, "porla_msm_resident");
    const int dev = device_init();
    std::lock_guard<std::mutex> lock(g_io_mu);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    MsmOptions opt;
    decode_plan(window_bits, &opt);
    opt.scalar_be = scalar_fmt == PORLA_SCALAR_BE32;
    opt.out_fmt = out_fmt;
    opt.shared_points = 1;
    static uint8_t* d_ws_dev[kMaxDevices] = {};  // 256 window sums of 128 B: more than any plan produces; one per device
    uint8_t*& d_ws = d_ws_dev[dev];
    if (!d_ws) PORLA_CUDA(cudaMalloc(&d_ws, 256 * 128));
    run_and_fetch(t->t.curve, t->t, (const uint8_t*)d_scalars, n, 1, opt, d_ws, (uint8_t*)h_out64, st);
}

void porla_msm_table_host_scalars_batch(const porla_table* t, int64_t first, const void* scalars, int64_t n, int64_t nbatch,
                                        int scalar_fmt, int out_fmt, void* out) {
    check_shape(n, nbatch, "porla_msm_table_host_scalars");
    if (first < 0 || n < 0 || nbatch < 0 || first + n > (int64_t)t->t.n) die("porla_msm_table_host_scalars: range outside the table");
    if (nbatch == 0) return;
    if (n == 0) {
        memset(out, 0, 64 * (size_t)nbatch);
        return;
    }
    device_init();
    StagedCall call(n, nbatch);
    const size_t sc_bytes = (size_t)n * nbatch * 32;
    call.add(sc_bytes);
    call.add_result(t->t.curve, n, nbatch);
    uint8_t* d = call.dev();
    h2d_copy(d, scalars, sc_bytes, call.stream());
    call.fetch(t->t.curve, table_window(t->t, first, n), d, n, nbatch, call.msm_options(scalar_fmt, out_fmt, 1), (uint8_t*)out);
}

void porla_msm_table_host_scalars(const porla_table* t, int64_t first, const void* scalars, int64_t n, int scalar_fmt,
                                  int out_fmt, void* out64) {
    porla_msm_table_host_scalars_batch(t, first, scalars, n, 1, scalar_fmt, out_fmt, out64);
}

void porla_msm_plan(int curve, int64_t n, int64_t nbatch, int window_bits, int* c_out, int* nwin_out) {
    MsmOptions o;
    decode_plan(window_bits, &o);
    MsmPlan p = msm_plan(curve, (uint32_t)n, (uint32_t)nbatch, o.window_bits, o.glv);
    *c_out = p.c | (p.glv ? PORLA_PLAN_GLV_ON : PORLA_PLAN_GLV_OFF);
    *nwin_out = p.nwin;
}

void porla_msm_window_sums_device(const porla_table* t, const void* d_scalars, int64_t n, int scalar_fmt, int window_bits,
                                  void* d_window_sums, void* cuda_stream) {
    check_shape(n, 1, "porla_msm_window_sums_device");
    if (n > (int64_t)t->t.n) die("porla_msm_window_sums_device: table shorter than the MSM");
    MsmOptions opt;
    decode_plan(window_bits, &opt);
    if (window_bits & PORLA_PLAN_FIXED) {   // the parts agreed on the expansion's window size: one sum per part
        if (t->t.fb_c <= 0 || t->t.fb_c != PORLA_PLAN_WINDOW(window_bits) || (int64_t)t->t.fb_n != (int64_t)t->t.n)
            die("porla_msm_window_sums_device: PORLA_PLAN_FIXED needs porla_table_precompute with the plan's window size");
        opt.window_bits = t->t.fb_c;
        opt.glv = 0;
        opt.no_small = 1;
    } else {
        const MsmPlan plan = msm_plan(t->t.curve, (uint32_t)n, 1, opt.window_bits, opt.glv);
        opt.window_bits = plan.c;
        opt.glv = plan.glv;
        opt.no_fixed_base = 1;  // the sharded protocol exchanges nwin window sums per rank
    }
    opt.scalar_be = scalar_fmt == PORLA_SCALAR_BE32;
    opt.shared_points = 1;
    opt.d_window_sums = d_window_sums;
    msm_device(t->t.curve, t->t, (const uint8_t*)d_scalars, (uint32_t)n, 1, opt, nullptr, nullptr, (cudaStream_t)cuda_stream);
}

void porla_msm_finalize_host(int curve, const void* h_window_sums, int64_t nparts, int nwin, int c, int out_fmt, void* out64) {
    finalize_host_parts(curve, h_window_sums, (int)nparts, nwin, PORLA_PLAN_WINDOW(c), out_fmt, (uint8_t*)out64);
}

void porla_msm_combine_device(int curve, const void* d_parts, int64_t count, int64_t nbatch, int out_fmt, void* d_out,
                              void* cuda_stream) {
    msm_combine_device(curve, d_parts, (uint32_t)count, (uint32_t)nbatch, out_fmt, (uint8_t*)d_out, (cudaStream_t)cuda_stream);
}

void porla_msm_host(int curve, const void* scalars, const void* points, int64_t n, int64_t nbatch, int scalar_fmt,
                    int point_fmt, void* out) {
    msm_host_core(curve, (const uint8_t*)scalars, (const uint8_t*)points, n, nbatch, scalar_fmt, point_fmt, (uint8_t*)out);
}

void porla_scalar_mul_batch_device(const porla_table* t, const void* d_scalars, int64_t n, int scalar_fmt, int out_fmt,
                                   void* d_out, void* cuda_stream) {
    check_shape(n, 1, "porla_scalar_mul_batch_device");
    if (t->t.n != 1 && n > (int64_t)t->t.n) die("porla_scalar_mul_batch_device: table shorter than the batch");
    device_init();
    cudaStream_t st = (cudaStream_t)cuda_stream;
    // A length-1 table that carries a look-up table (porla_table_precompute with window_bits = 0) is a fixed base: each
    // product is a sum of nwin table entries.  Every other table keeps the double-and-add of k_scalar_mul; that includes
    // the generator table of porla_table_create_multiples, which is imported without a look-up table.  Both paths return
    // canonical points, so the bytes do not depend on the path.
    if (t->t.n == 1 && t->t.d_lut) {
        fixed_base_mul_device(t->t.curve, t->t, (const uint8_t*)d_scalars, scalar_fmt == PORLA_SCALAR_BE32, (uint32_t)n, out_fmt,
                              (uint8_t*)d_out, st);
        return;
    }
    void* d_aff = nullptr;
    PORLA_CUDA(cudaMallocAsync(&d_aff, (size_t)(n ? n : 1) * 64, st));
    scalar_mul_device(t->t.curve, t->t, (const uint8_t*)d_scalars, scalar_fmt == PORLA_SCALAR_BE32, (uint32_t)n, d_aff, st);
    export_points_device(t->t.curve, d_aff, (uint32_t)n, out_fmt, (uint8_t*)d_out, st);
    PORLA_CUDA(cudaFreeAsync(d_aff, st));
}

void bn254_align_mac_batch(GoSlice* data, GoInt batch, GoSlice* align_out) {
    const int64_t n = g_kzg.n_samples;
    if (batch < 0 || data->len < batch * n * 64) die("bn254_align_mac_batch: data shorter than batch*n_samples*64 bytes");
    if (batch == 0) return;
    check_shape(n, batch, "bn254_align_mac_batch");
    device_init();
    std::shared_lock<std::shared_mutex> srs = srs_reader(n, 0, batch);   // also refuses n_samples above the SRS length
    std::vector<uint8_t> res((size_t)batch * 64);
    align_mac_core(kCurveBn254, g_kzg.srs_table, data->data, n, batch, PORLA_POINT_BE64, res.data());
    go_copy(align_out, res.data(), res.size());
}

void bn254_audit_aggregate(GoSlice* coefs, GoSlice* blocks, GoInt n, GoSlice* b_out, GoSlice* align_out) {
    const int64_t chunks = g_kzg.n_samples;
    if (n < 0 || n >= (1 << 24)) die("bn254_audit_aggregate: block count out of range");
    if (coefs->len < n * 4 || blocks->len < n * chunks * 64) die("bn254_audit_aggregate: coefs / blocks shorter than n entries");
    check_shape(chunks, 1, "bn254_audit_aggregate");
    device_init();
    std::shared_lock<std::shared_mutex> srs = srs_reader(chunks, 0, 1);   // also refuses n_samples above the SRS length
    std::vector<uint8_t> b_mod((size_t)chunks * 32), res(64);
    audit_aggregate_core(kCurveBn254, g_kzg.srs_table, coefs->data, blocks->data, n, chunks, PORLA_POINT_BE64, b_mod.data(),
                         res.data());
    go_copy(b_out, b_mod.data(), b_mod.size());
    go_copy(align_out, res.data(), res.size());
}

void porla_data_butterfly_stage(void* blocks, int64_t n_blocks, int64_t chunks, int64_t m, const void* twiddles_le32,
                                const void* lcm_le64) {
    if (m < 2 || (m & (m - 1)) || n_blocks % m || chunks <= 0) die("porla_data_butterfly_stage: m must be a power of two dividing the block count");
    device_init();
    StagedCall call;
    const size_t bytes = (size_t)n_blocks * chunks * 64, tw_bytes = (size_t)(m / 2) * 32;
    call.add(bytes);
    const size_t tw_off = call.add(tw_bytes);
    uint8_t* d = call.dev();
    cudaStream_t st = call.stream();
    h2d_copy(d, blocks, bytes, st);
    PORLA_CUDA(cudaMemcpyAsync(d + tw_off, twiddles_le32, tw_bytes, cudaMemcpyHostToDevice, st));
    data_butterfly_stage_device(reinterpret_cast<uint32_t*>(d), (uint32_t)n_blocks, (uint32_t)chunks, (uint32_t)m, d + tw_off,
                                (const uint8_t*)lcm_le64, st);
    PORLA_CUDA(cudaMemcpyAsync(blocks, d, bytes, cudaMemcpyDeviceToHost, st));
    PORLA_CUDA(cudaStreamSynchronize(st));
}

void porla_data_butterfly_stage_device(void* d_blocks, int64_t n_blocks, int64_t chunks, int64_t m, const void* d_twiddles_le32,
                                       const void* lcm_le64, void* cuda_stream) {
    if (m < 2 || (m & (m - 1)) || n_blocks % m || chunks <= 0) die("porla_data_butterfly_stage_device: m must be a power of two dividing the block count");
    data_butterfly_stage_device(reinterpret_cast<uint32_t*>(d_blocks), (uint32_t)n_blocks, (uint32_t)chunks, (uint32_t)m,
                                (const uint8_t*)d_twiddles_le32, (const uint8_t*)lcm_le64, (cudaStream_t)cuda_stream);
}

void porla_butterfly_stage_device(porla_table* t, int64_t m, const void* twiddles, int scalar_fmt, int twiddles_on_device,
                                  void* cuda_stream) {
    if (m < 2 || (m & (m - 1)) || (int64_t)t->t.n % m) die("porla_butterfly_stage_device: m must be a power of two dividing the table length");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const uint8_t* d_tw = (const uint8_t*)twiddles;
    uint8_t* d_tmp = nullptr;
    if (!twiddles_on_device) {
        PORLA_CUDA(cudaMallocAsync(&d_tmp, (size_t)(m / 2) * 32, st));
        PORLA_CUDA(cudaMemcpyAsync(d_tmp, twiddles, (size_t)(m / 2) * 32, cudaMemcpyHostToDevice, st));
        d_tw = d_tmp;
    }
    butterfly_stage_device(&t->t, (uint32_t)m, d_tw, scalar_fmt == PORLA_SCALAR_BE32, st);
    if (d_tmp) {
        PORLA_CUDA(cudaFreeAsync(d_tmp, st));
        PORLA_CUDA(cudaStreamSynchronize(st));   // the host twiddle buffer may be reused by the caller
    }
}

}  // extern "C"

namespace porla {
// A stage of at most this many butterflies runs on the calling host (up to 8 threads), like the single-point symbols it
// replaces: one butterfly is a dependent chain of ~127 doublings and additions, 1.4 ms on one GPU thread against 0.1 ms on a
// host core, so the device only wins once there are enough butterflies to fill it (measured with tools/replay_config1:
// Porla's per-update hierarchy rebuilds issue stages of 1 .. 512 butterflies).  secp256k1 crosses over sooner: its host
// stage takes 0.39 / 0.92 ms at 32 / 64 butterflies against ~0.56 ms for a stage through the device (one B200, 1000 W;
// tools/secp_butterfly_times.py).  PORLA_HOST_BUTTERFLIES overrides (0: always device).
int64_t host_butterfly_limit(int curve) {
    const char* e = getenv("PORLA_HOST_BUTTERFLIES");
    return e ? (int64_t)atoll(e) : (curve == kCurveBn254 ? (int64_t)96 : (int64_t)32);
}

void for_each_butterfly_host(int64_t nb, const std::function<void(int64_t, int64_t)>& body) {
    const int64_t nt = nb >= 16 ? 8 : (nb >= 4 ? 4 : 1);
    if (nt == 1) {
        body(0, nb);
        return;
    }
    std::vector<std::thread> th;
    for (int64_t t = 0; t < nt; t++) th.emplace_back(body, nb * t / nt, nb * (t + 1) / nt);
    for (auto& x : th) x.join();
}
}  // namespace porla

static void butterfly_stage_host(uint8_t* pts, int64_t n, int64_t m, const uint8_t* tw) {
    const int64_t m2 = m / 2;
    for_each_butterfly_host(n / 2, [&](int64_t lo, int64_t hi) {
        for (int64_t b = lo; b < hi; b++) {
            const int64_t j = b % m2, k = (b / m2) * m + j;
            G1A a0 = G1A::inf(), a1 = G1A::inf();
            g1_unmarshal(pts + 64 * k, 64, &a0);
            g1_unmarshal(pts + 64 * (k + m2), 64, &a1);
            const G1A t = g1_mul(a1, elem_from_be<Fr>(tw + 32 * j, 32));
            g1_marshal(g1_add(a0, t), pts + 64 * k);
            g1_marshal(g1_add(a0, t.neg()), pts + 64 * (k + m2));
        }
    });
}

extern "C" {

void bn254_butterfly_stage(GoSlice* points, GoInt n, GoInt m, GoSlice* twiddles) {
    if (n < 0 || points->len < n * 64 || twiddles->len < (m / 2) * 32)
        die("bn254_butterfly_stage: slices shorter than n points / m/2 twiddles");
    if (m < 2 || (m & (m - 1)) || n % m) die("bn254_butterfly_stage: m must be a power of two dividing n");
    if (n == 0) return;
    check_shape(n, 1, "bn254_butterfly_stage");
    if (n / 2 <= host_butterfly_limit(kCurveBn254)) {
        butterfly_stage_host((uint8_t*)points->data, n, m, (const uint8_t*)twiddles->data);
        return;
    }
    device_init();
    StagedCall call;
    porla_table t;
    table_import_host(kCurveBn254, (const uint8_t*)points->data, PORLA_POINT_BE64, (uint32_t)n, &t.t, call.stream());
    porla_butterfly_stage_device(&t, m, twiddles->data, PORLA_SCALAR_BE32, 0, call.stream());
    porla_table_export(&t, PORLA_POINT_BE64, points->data, 0, call.stream());
    table_free(&t.t);
}

int porla_debug_pairing_selfcheck(int rounds) {
    // Host-only consistency check of the verifier's pairing: for random a, b
    //   e(aG1, bG2) * e(-(ab)G1, G2) == 1   and   e(aG1, bG2) * e(-(ab + 1)G1, G2) != 1
    // under BOTH hard-part routines (the u-addition chain used in production and the plain 761-bit
    // exponentiation), and the lockstep multi-pairing Miller loop agrees with the product of single loops.
    int bad = 0;
    std::mt19937_64 rng(12345);
    G1A g1 = g1_generator();
    G2A g2 = g2_generator();
    for (int it = 0; it < rounds; it++) {
        uint8_t ab[32], bb[32];
        for (int i = 0; i < 32; i++) {
            ab[i] = (uint8_t)rng();
            bb[i] = (uint8_t)rng();
        }
        Fr a = elem_from_be<Fr>(ab, 32), b = elem_from_be<Fr>(bb, 32);
        G1A pa = g1_mul(g1, a);
        G2A qb = g2_mul(g2, b);
        G1A pab = g1_mul(g1, a * b).neg();
        G1A pab1 = g1_mul(g1, a * b + Fr::one()).neg();
        for (int wrong = 0; wrong < 2; wrong++) {
            G1A ps[2] = {pa, wrong ? pab1 : pab};
            G2A qs[2] = {qb, g2};
            Fq12 m = miller_loop_multi(ps, qs, 2);
            Fq12 m2 = miller_loop(ps[0], qs[0]).mul_dense(miller_loop(ps[1], qs[1]));
            Fq12 e1 = m.conj6().mul_dense(fq12_inv(m));
            Fq12 e2 = m2.conj6().mul_dense(fq12_inv(m2));
            Fq12 c1 = frob2(e1).mul_dense(e1), c2 = frob2(e2).mul_dense(e2);
            bool chain1 = hard_part_chain(c1).is_one(), plain1 = hard_part_plain(c1).is_one();
            bool chain2 = hard_part_chain(c2).is_one(), plain2 = hard_part_plain(c2).is_one();
            bool expect = wrong == 0;
            if (chain1 != expect || plain1 != expect || chain2 != expect || plain2 != expect) bad++;
            // c1 lies in the cyclotomic subgroup (easy part done): the Granger-Scott squaring must equal the generic one
            Fq12 g = c1;
            for (int rep = 0; rep < 3; rep++) {
                Fq12 s1 = fq12_cyclotomic_sqr(g), s2 = g.sqr();
                for (int k = 0; k < 6; k++)
                    if (!(s1.c[k] == s2.c[k])) {
                        bad++;
                        break;
                    }
                g = s2.mul_dense(c2);
            }
            // the fixed-argument loop (precomputed lines of qb and g2) must give the very same Fp12 value
            G2Lines la = g2_precompute_lines(qb), lb = g2_precompute_lines(g2);
            const G2Lines* ls[2] = {&la, &lb};
            Fq12 mf = miller_loop_fixed(ps, ls, 2);
            bool same = la.valid && lb.valid;
            for (int k = 0; k < 6 && same; k++) same = mf.c[k] == m.c[k];
            if (!same) bad++;
        }
    }
    return bad;
}

void porla_debug_field_op(int curve, int op, const void* a, const void* b, int64_t n, void* out) {
    device_init();
    StagedCall call;
    const size_t bytes = (size_t)n * 32, a_off = call.add(bytes), b_off = call.add(bytes), out_off = call.add(bytes);
    uint8_t* d = call.dev();
    cudaStream_t st = call.stream();
    PORLA_CUDA(cudaMemcpyAsync(d + a_off, a, bytes, cudaMemcpyHostToDevice, st));
    PORLA_CUDA(cudaMemcpyAsync(d + b_off, b, bytes, cudaMemcpyHostToDevice, st));
    field_mul_device(curve, d + a_off, d + b_off, (uint32_t)n, op, d + out_off, st);
    PORLA_CUDA(cudaMemcpyAsync(out, d + out_off, bytes, cudaMemcpyDeviceToHost, st));
    PORLA_CUDA(cudaStreamSynchronize(st));
}

void porla_debug_field_mul(int curve, const void* a, const void* b, int64_t n, void* out) {
    porla_debug_field_op(curve, 0, a, b, n, out);
}

}  // extern "C"
