// Host-side interface of the device MSM engine (internal to libmultiexp.so; the public C-ABI is
// include/porla_multiexp.h).  One engine per (process, device, curve); calls are serialised by
// an internal mutex because Porla invokes the C-ABI from up to 8 pool threads
// (/root/reference/porla/Server/Server.hpp:1077-1078).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace porla {

enum CurveId : int { kCurveBn254 = 0, kCurveSecp256k1 = 1 };

// Throws nothing; every failure is fatal by design ("no CPU fallback"): prints and aborts.
void cuda_check(cudaError_t e, const char* what, const char* file, int line);
#define PORLA_CUDA(x) ::porla::cuda_check((x), #x, __FILE__, __LINE__)

// Selects/initialises the process's default device once (PORLA_DEVICE, else LOCAL_RANK, else 0) and makes the calling
// thread's device current: the default one, or the one a DeviceScope on this thread names.  Aborts loudly when no CUDA
// device is usable.
int device_init();
// Non-aborting probe (lets the host-only entry points of the C-ABI work on a machine without a GPU).
bool device_available();
constexpr int kMaxDevices = 16;   // devices one process drives at most
int device_count();          // visible CUDA devices (0 when there is none)
int default_device();        // the device a plain call runs on (after device_init)
int current_device();        // the calling thread's engine device: its DeviceScope's, else the default one
// true when the process was told which ONE device is its own (PORLA_DEVICE / LOCAL_RANK set: one process per GPU under
// torchrun); an in-call fan-out over all visible devices is then opt-in (PORLA_DEVICES) instead of automatic.
bool device_pinned_by_env();
// Every engine object (scratch arena, engine mutex, stage timer) exists once per device; a thread that works on
// another device than the default one (the in-call multi-GPU partition, Client.hpp:747-787) holds a DeviceScope.
struct DeviceScope {
    int prev;
    explicit DeviceScope(int dev);
    ~DeviceScope();
    DeviceScope(const DeviceScope&) = delete;
    DeviceScope& operator=(const DeviceScope&) = delete;
};

// Resident point table in internal form (Montgomery for BN254).
struct PointTable {
    void* d_points = nullptr;     // Affine<F>[n]
    uint8_t* d_flags = nullptr;   // 1 = infinity; nullptr when the table has none
    uint32_t n = 0;
    uint32_t n_inf = 0;
    int curve = 0;
    // Optional fixed-base expansion (table_precompute): fb_points[w*n + i] = 2^(fb_c*w) * P_i for
    // w < fb_nwin.  With it, every window of an MSM over this table shares ONE bucket set: no
    // per-window bucket reduction and no doublings in the window combine.
    int fb_c = 0;
    int fb_nwin = 0;
    uint32_t fb_n = 0;            // row stride of the expansion = length of the table it was built for (a view
                                  // [first, first + n) of the table keeps it and offsets the pointers by `first`)
    void* d_fb_points = nullptr;
    // Optional look-up table of EVERY window multiple on top of the expansion (small tables only):
    // lut[((i*fb_nwin + w) << (fb_c-1)) + d - 1] = d * 2^(fb_c*w) * P_i, 1 <= d <= 2^(fb_c-1).  An MSM over the
    // table is then a plain sum of n * fb_nwin entries (k_lut_sum): no sort, no buckets, no doublings.
    void* d_lut = nullptr;
    // GLV (BN254): the endomorphism image phi(P_i) = (beta x_i, y_i) of every entry.  Only beta x_i is stored (32 B per
    // point, d_phi_x, right behind the table; y_i is read from the table itself), so table + image are 96 B per point.
    // A (point, window) pair addresses phi(P_i) as index phi_off + i (0 = image absent; every import path of a GLV
    // curve writes it, the butterfly kernel refreshes it).
    uint32_t phi_off = 0;
    void* d_phi_x = nullptr;
};

// Import `n` external 64-byte points that already live on the device.
void table_import_device(int curve, const uint8_t* d_bytes, int point_fmt, uint32_t n, PointTable* out,
                         cudaStream_t stream);
// Import from host memory (H2D copy + conversion).
void table_import_host(int curve, const uint8_t* h_bytes, int point_fmt, uint32_t n, PointTable* out,
                       cudaStream_t stream);
void table_free(PointTable* t);
// Builds the fixed-base expansion for window size c (0 = choose for MSMs of `n_hint` terms, `batch_hint`
// per launch).  One-time cost of ~254 doublings + fb_nwin inversions per point; fb_nwin * n * 64 bytes.
int table_precompute(PointTable* t, int c, uint32_t n_hint, uint32_t batch_hint, cudaStream_t stream);
int choose_window_fixed_base(int curve, uint32_t n, uint32_t nbatch);
// Import into caller-provided device buffers (2*n*64 B points: the table and its endomorphism image, n B flags):
// no allocation, no sync.  The returned table borrows the buffers (do not table_free it).
void table_import_into(int curve, const uint8_t* d_bytes, int point_fmt, uint32_t n, void* d_points_out,
                       uint8_t* d_flags_out, PointTable* out, cudaStream_t stream, bool with_phi = true);
// Import `n` secp256k1 Jacobian points (IPA-mode MACs) into caller-provided device buffers (n * 64 B points, n B flags):
// d_xyz holds canonical X, Y, Z (8 LE 32-bit limbs each), d_inf their infinity flags; one inversion per point with Z != 1.
// No allocation, no sync.  The returned table borrows the buffers (do not table_free it).
void table_import_jacobian_secp256k1(const uint32_t* d_xyz, const uint8_t* d_inf, uint32_t n, void* d_points_out,
                                     uint8_t* d_flags_out, PointTable* out, cudaStream_t stream);

struct MsmOptions {
    int window_bits = 0;      // 0 = choose from n
    int scalar_be = 1;        // 1: 32-byte big-endian scalars, 0: 8 LE 32-bit limbs
    int out_fmt = 0;          // PointFormat of the serialised result
    int shared_points = 1;    // batch: all MSMs over the same table prefix
    // When set, receives the nbatch*nwin per-window sums (XYZZ, 128 B each, window-major per MSM)
    // and the device finaliser is skipped: the caller combines them with finalize_host().
    void* d_window_sums = nullptr;
    int no_fixed_base = 0;    // ignore the table's fixed-base expansion (callers that need nwin window sums)
    // Upper bound on the bit length of every (reduced) scalar when the caller knows it (the legacy C-ABI scans
    // its host buffer: Porla's audit coefficients are 31-bit, utils.h:271-275); 0 = the full order width.
    int max_scalar_bits = 0;
    int no_small = 0;         // always run the sort / accumulate / reduce pipeline
    int glv = -1;             // -1: decided by the plan; 0 / 1: forced (parts of one MSM must agree on the window layout)
    // Caller-owned device scratch for the one-launch small paths: when it is large enough the call takes neither the
    // engine's arena nor its mutex, so small MSMs issued from several host threads (Porla's pool of 8,
    // Server.hpp:1077-1078) run concurrently on their own streams.
    void* d_scratch = nullptr;
    size_t scratch_bytes = 0;
    // Streamed MSM (multi.cu: msm_host_pipelined): the terms arrive in parts, every part is recoded, sorted and accumulated
    // by its own call INTO ONE shared bucket array, and only the last call reduces the buckets.  part_mode: 0 a whole MSM,
    // 1 first part (clears the buckets), 2 middle part, 3 last part (accumulates, then reduces).  d_buckets: the shared
    // array, msm_bucket_bytes() bytes; every part must use the same window layout (window_bits and glv forced).
    int part_mode = 0;
    void* d_buckets = nullptr;
};
enum : int { kPartWhole = 0, kPartFirst = 1, kPartMiddle = 2, kPartLast = 3 };

enum PlanMode : int { kPlanPipeline = 0, kPlanBits = 1, kPlanLut = 2 };
struct MsmPlan {
    int c;      // window bits
    int nwin;   // window sums per MSM handed to the finaliser
    int mode;   // PlanMode
    int glv;    // pipeline only: scalars split with the GLV endomorphism; nwin then counts the windows of ONE half
};
// The sort / accumulate / reduce pipeline's plan for n terms.
MsmPlan msm_plan(int curve, uint32_t n, uint32_t nbatch, int window_bits, int glv = -1);
// Bytes of the bucket array of ONE MSM under a pipeline plan (nwin bucket sets of 2^(c-1) XYZZ records).
size_t msm_bucket_bytes(const MsmPlan& plan);
// Plan for a specific call.  Fixed-base expansion applicable: nwin = 1 (a single shared bucket set or the
// look-up table, one "window sum" per MSM, no doublings), c = the expansion's window size.  Few terms in
// total and no explicit window size: one window per scalar bit (k_small_bits), c = 1.
MsmPlan msm_plan_table(const PointTable& t, uint32_t n, uint32_t nbatch, const MsmOptions& opt);

// Host-side tail of one MSM: Horner over the window sums (c doublings per window), affine
// normalisation, serialisation.  h_window_sums: nwin XYZZ records as produced on the device.
void finalize_host(int curve, const void* h_window_sums, int nwin, int c, int out_fmt, uint8_t* out64);
// Same for an MSM sharded over `nparts` devices: h_window_sums holds nparts consecutive sets of
// nwin window sums (all computed with the same window size); they are added window by window.
void finalize_host_parts(int curve, const void* h_window_sums, int nparts, int nwin, int c, int out_fmt, uint8_t* out64);

// nbatch MSMs of n terms each.  d_scalars: nbatch*n*32 bytes on the device.
// d_out (nullable): nbatch*64 bytes, canonical affine.  d_out_xyzz (nullable): nbatch*128 bytes,
// un-normalised sums in internal form (for multi-GPU combination).
void msm_device(int curve, const PointTable& table, const uint8_t* d_scalars, uint32_t n,
                uint32_t nbatch, const MsmOptions& opt, uint8_t* d_out, void* d_out_xyzz,
                cudaStream_t stream);

// Sum `count` XYZZ partials per MSM (layout parts[k*nbatch + m]) and serialise nbatch results.
void msm_combine_device(int curve, const void* d_parts, uint32_t count, uint32_t nbatch, int out_fmt,
                        uint8_t* d_out, cudaStream_t stream);

// Elementwise batched kernels.
void scalar_mul_device(int curve, const PointTable& table, const uint8_t* d_scalars, int scalar_be,
                       uint32_t n, void* d_out_affine, cudaStream_t stream);
// out[i] = k_i * B for the ONE base of `table`, which must be a length-1 table carrying a look-up table (table_precompute
// with window_bits = 0): a sum of nwin table entries per scalar, no doublings.  d_out: n * 64 B, canonical affine in out_fmt.
void fixed_base_mul_device(int curve, const PointTable& table, const uint8_t* d_scalars, int scalar_be, uint32_t n, int out_fmt,
                           uint8_t* d_out, cudaStream_t stream);
// out[b] = sum_i f_(b,i) * powers[i] mod r (BN254 scalar field) for nbatch records of n big-endian 32-byte coefficients,
// each reduced mod r first (fr.Element.SetBytes); d_powers: n field elements in Montgomery form (Fp<Bn254FrParams>).
// d_out: nbatch canonical scalars of 8 little-endian 32-bit limbs (PORLA_SCALAR_LE32).
void fr_poly_eval_device(const uint8_t* d_coeffs_be, const void* d_powers, uint32_t n, uint32_t nbatch, uint8_t* d_out,
                         cudaStream_t stream);
// One radix-2 butterfly stage of the "FFT in the exponent", in place on a resident table whose length is a
// multiple of m (m a power of two >= 2): see k_butterfly.  d_twiddles: m/2 scalars of 32 bytes on the device.
// Invalidates the table's fixed-base expansion.
void butterfly_stage_device(PointTable* t, uint32_t m, const uint8_t* d_twiddles, int scalar_be, cudaStream_t stream);
// Server::align_MAC's scalar preparation for `total` chunks of 64 bytes (16 LE limbs, values below
// PRIME_MODULUS * r): chunk <- chunk % PRIME_MODULUS in place, scalars_be[i] = (chunk % PRIME_MODULUS - chunk) % r,
// r the group order of `curve` (BN254 in KZG mode, secp256k1 in IPA mode).
void align_scalars_device(int curve, uint32_t* d_data, uint32_t total, uint8_t* d_scalars_be, cudaStream_t stream);
// Server::audit's aggregation of `n` data blocks of `chunks` 64-byte chunks (16 LE limbs) with 31-bit coefficients,
// followed by align_MAC's arithmetic on the sums: b_mod_be[j] = B_j % PRIME_MODULUS and
// c_be[j] = (B_j % PRIME_MODULUS - B_j) % r as 32-byte big-endian scalars, B_j = sum_i coefs[i] * blocks[i][j].
void audit_aggregate_device(int curve, const uint32_t* d_coefs, const uint32_t* d_blocks, uint32_t n, uint32_t chunks,
                            uint8_t* d_b_mod_be, uint8_t* d_c_be, cudaStream_t stream);
// One radix-2 stage of the FFT on the data blocks themselves (Server.hpp:1582-1588): n_blocks x chunks chunks of 64 bytes
// (16 LE limbs, values below lcm), in place; twiddles: m/2 scalars of 32 bytes, little-endian; lcm_le64: the modulus
// (utils.h:42-43), whose Barrett constant is derived on the host per call.
void data_butterfly_stage_device(uint32_t* d_blocks, uint32_t n_blocks, uint32_t chunks, uint32_t m, const uint8_t* d_twiddles,
                                 const uint8_t* lcm_le64, cudaStream_t stream);
void export_points_device(int curve, const void* d_affine, uint32_t n, int point_fmt, uint8_t* d_out,
                          cudaStream_t stream);
void field_mul_device(int curve, const void* d_a, const void* d_b, uint32_t n, int op, void* d_out,
                      cudaStream_t stream);

// Per-stage CUDA-event timing of the most recent msm_device call (count, scan, scatter, accumulate,
// reduce, finalize), in ms.  Returns the number of stages written (0 when disabled).
void stage_timing_enable(int on);
int stage_timing_read(float* ms_out);

int choose_window(int curve, uint32_t n, uint32_t nbatch);
uint64_t launches_issued();   // number of kernels this library has launched (bench's gpu_launches)

}  // namespace porla
