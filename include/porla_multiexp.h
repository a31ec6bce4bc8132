/* porla_multiexp.h -- C-ABI of the B200-native libmultiexp.so
 *
 * Part 1 is byte-for-byte the contract of the cgo-generated header the Porla C++ code includes
 * today (/root/reference/porla/Utils/libmultiexp.h:61 GoSlice, :71-84 the 14 prototypes; Go side
 * /root/reference/porla/main.go).  A Porla Client/Server built with ENABLE_KZG links against this
 * library unchanged (-lmultiexp, /root/reference/porla/Makefile:13).
 *
 * Part 2 adds what the reference lacks and BASELINE.json's north star asks for: batched MSM entry
 * points, device-resident tables/MSMs for callers that keep data in HBM, and the secp256k1
 * (IPA mode) multi-exponentiation behind the signature of secp256k1_ecmult_multi_var
 * (/root/reference/porla/Utils/secp256k1_lib/ecmult.h:34-48).
 *
 * All MSMs run on the GPU (sm_100a).  There is no CPU fallback: without a usable CUDA device
 * every MSM entry point prints a diagnostic and aborts.  Single-point operations (add_point,
 * mult_point, neg_point, ...) and the KZG verifier's pairing are O(1) work per call and run in
 * host C++ inside this library.
 */
#ifndef PORLA_MULTIEXP_H
#define PORLA_MULTIEXP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ Part 1: legacy cgo ABI */
#ifndef GO_CGO_PROLOGUE_H
#define GO_CGO_PROLOGUE_H
typedef signed char GoInt8;
typedef unsigned char GoUint8;
typedef long long GoInt64;
typedef unsigned long long GoUint64;
typedef GoInt64 GoInt;
typedef GoUint64 GoUint;
typedef struct { void *data; GoInt len; GoInt cap; } GoSlice; /* libmultiexp.h:61 */
#endif

/* main.go:32   tau and alpha: big-endian integers of any length, reduced mod r. */
extern void init_key(GoSlice* tau_key_in, GoSlice* alpha_key_in);
/* main.go:43   SRS = {[tau^i]G1 (i < SRS_size), [1]G2, [tau]G2}; blob = 2x64 B compressed G2 +
 *              4 B BE count + SRS_size x 32 B compressed G1 (4228 B for 128); also draws h_MAC.
 *              Uploads the G1 bases to HBM. */
extern void init_SRS(GoInt SRS_size, GoSlice* out, GoInt64* out_len);
/* main.go:63   parse the blob produced by init_SRS, upload the G1 bases to HBM. */
extern void init_SRS_from_data(GoInt SRS_size, GoSlice* in);
/* main.go:71   [alpha * f(tau)] G1 via Horner (trapdoor shortcut, no MSM). */
extern void compute_digest(GoSlice* data_in, GoSlice* data_out);
/* main.go:92   [s] h_MAC. */
extern void compute_digest_complement(GoSlice* data_in, GoSlice* data_out);
/* main.go:104  kzg.Commit: n_samples-term fixed-base MSM over the resident SRS (GPU). */
extern void compute_digest_from_srs(GoSlice* data_in, GoSlice* data_out);
/* main.go:119  general G1 MSM: scalars length x 32 B BE (reduced mod r), points length x 64 B
 *              gnark Marshal layout, result 64 B (GPU). */
extern void compute_multi_exp(GoSlice* scalars, GoSlice* points, GoInt length, GoSlice* result_out);
/* main.go:141 */
extern GoUint8 compare_commitment(GoSlice* commitment_a, GoSlice* commitment_b);
/* main.go:154  C = Commit(f); y = f(z); H = Commit((f - y)/(X - z))  (two GPU MSMs). */
extern void create_proof(GoUint64 random_point, GoSlice* data_in, GoSlice* commitment_out,
                         GoSlice* proof_H, GoSlice* proof_point, GoSlice* proof_claim);
/* main.go:178  e(C - [y]G1, G2) * e(-H, [tau]G2 - [z]G2) == 1. */
extern GoUint8 verify_proof(GoSlice* commitment_in, GoSlice* proof_H, GoSlice* proof_point,
                            GoSlice* proof_claim);
/* main.go:196-230  in-place single-point operations on 64-byte buffers. */
extern void add_point(GoSlice* point_a, GoSlice* point_b);
extern void mult_point(GoSlice* point_a, GoSlice* scalar);
extern void neg_point(GoSlice* point);
extern void set_inf_point(GoSlice* point);

/* ------------------------------------------------------------------ Part 2: new entry points */
enum { PORLA_CURVE_BN254 = 0, PORLA_CURVE_SECP256K1 = 1 };
enum { PORLA_SCALAR_BE32 = 0,   /* 32-byte big-endian integer (bn254_scalar, utils.h:307-318) */
       PORLA_SCALAR_LE32 = 1 }; /* 8 little-endian 32-bit limbs (secp256k1_scalar, scalar_4x64.h:13) */
enum { PORLA_POINT_BE64 = 0,    /* X||Y big-endian (gnark Marshal; SEC1 uncompressed minus the tag) */
       PORLA_POINT_LE64 = 1 };  /* x,y as 8 little-endian 32-bit limbs each, canonical */

/* Selects the CUDA device (PORLA_DEVICE, else LOCAL_RANK, else 0); returns its index.
 * Aborts loudly if there is none. */
int porla_device_init(void);
/* Kernels launched by this library so far (bench.py's gpu_launches). */
uint64_t porla_launch_count(void);

/* Batched forms of the two MSM entry points (many MSMs per launch sequence).
 * compute_multi_exp_batch: `batch` independent MSMs of `length` terms, scalars batch*length*32 B,
 * points batch*length*64 B, results batch*64 B.
 * compute_digest_from_srs_batch: `batch` coefficient vectors of n_samples*32 B over the resident
 * SRS (Porla's per-block commitments / align_MAC, Server.hpp:550-558), results batch*64 B. */
extern void compute_multi_exp_batch(GoSlice* scalars, GoSlice* points, GoInt length, GoInt batch,
                                    GoSlice* results_out);
extern void compute_digest_from_srs_batch(GoSlice* data_in, GoInt batch, GoSlice* data_out);
/* Batched forms of the client's two KZG symbols: each record is byte-identical to the per-call symbol on that record.
 * compute_digest_batch: data_in = batch * n_samples * 32 B of big-endian coefficients (each reduced mod r), data_out =
 * batch * 64 B of [alpha * f(tau)]G1.  alpha * f(tau) is evaluated on the device over powers alpha * tau^i kept in HBM,
 * the product runs over a resident look-up table of the digest base; both are rebuilt after init_key / init_SRS*.
 * compute_digest_complement_batch: data_in = batch * 32 B big-endian scalars s_i, each reduced mod r (the per-call
 * compute_digest_complement reads one scalar of any length), data_out = batch * 64 B of [s_i]h_MAC, over a resident
 * look-up table of h_MAC rebuilt after every init_SRS (before any init_SRS, h_MAC is infinity: 64 zero bytes per record).
 * batch == 0 returns without touching the device.  The per-call symbols stay on the host. */
extern void compute_digest_batch(GoSlice* data_in, GoInt batch, GoSlice* data_out);
extern void compute_digest_complement_batch(GoSlice* data_in, GoInt batch, GoSlice* data_out);

/* Resident point tables ("SRS and generator tables resident in HBM, uploaded once"). */
typedef struct porla_table porla_table;
porla_table* porla_table_create(int curve, const void* points, int64_t n, int point_fmt,
                                int on_device, void* cuda_stream);
/* table[i] = k_i * G (generator), k_i 32-byte scalars; used to build synthetic inputs whose MSM
 * has a closed form. */
porla_table* porla_table_create_multiples(int curve, const void* scalars, int64_t n, int scalar_fmt,
                                          int on_device, void* cuda_stream);
/* Fixed-base expansion of a resident table: stores 2^(c*w) * P_i for every window w (nwin * n * 64 B
 * of HBM, one-time ~254 doublings per point).  MSMs over the table (shared_points, window_bits 0 or
 * equal to the returned c) then use ONE bucket set for all windows: no per-window bucket reduction
 * and no doublings in the window combine.  window_bits 0 = choose for MSMs of n_hint terms, batch_hint
 * per launch.  Meant for the SRS / generator tables; arbitrary per-call points use the general path. */
int porla_table_precompute(porla_table* t, int window_bits, int64_t n_hint, int64_t batch_hint, void* cuda_stream);
int64_t porla_table_len(const porla_table* t);
int64_t porla_table_num_infinity(const porla_table* t);
void porla_table_export(const porla_table* t, int point_fmt, void* out, int on_device, void* cuda_stream);
void porla_table_destroy(porla_table* t);

/* nbatch MSMs of n terms over a resident table, scalars and results in device memory.
 * shared_points != 0: every MSM uses table[0..n); else MSM m uses table[m*n..(m+1)*n).
 * window_bits 0 = automatic.  d_out (nullable): nbatch*64 B canonical affine in out_fmt.
 * d_out_xyzz (nullable): nbatch*128 B un-normalised partial sums for porla_msm_combine_device.
 * Asynchronous on cuda_stream. */
void porla_msm_device(const porla_table* t, const void* d_scalars, int64_t n, int64_t nbatch,
                      int scalar_fmt, int shared_points, int window_bits, int out_fmt, void* d_out,
                      void* d_out_xyzz, void* cuda_stream);
/* One MSM over table[0..n) with device-resident scalars and the 64-byte result delivered to HOST
 * memory (synchronous).  The data-parallel stages run on the GPU; the serial tail -- Horner over
 * the <= 64 per-window sums and the affine normalisation -- runs on the calling host thread
 * (set PORLA_DEVICE_FINALIZE=1 to keep it on the device). */
void porla_msm_resident(const porla_table* t, const void* d_scalars, int64_t n, int scalar_fmt,
                        int window_bits, int out_fmt, void* h_out64, void* cuda_stream);
/* One MSM over table[first .. first + n) with HOST scalars (n x 32 bytes) and the 64-byte result in host
 * memory: the resident-generator form of compute_multi_exp (only the scalars cross PCIe). */
void porla_msm_table_host_scalars(const porla_table* t, int64_t first, const void* scalars, int64_t n,
                                  int scalar_fmt, int out_fmt, void* out64);
/* The same for `nbatch` scalar vectors over the same range in one launch (scalars nbatch*n*32 B, out nbatch*64 B):
 * the L and R of one inner-product round, which depend on the same challenge. */
void porla_msm_table_host_scalars_batch(const porla_table* t, int64_t first, const void* scalars, int64_t n,
                                        int64_t nbatch, int scalar_fmt, int out_fmt, void* out);
/* Building blocks of a range-sharded MSM (one process per GPU, SURVEY.md 8(e)): every rank runs
 * the pipeline over its point range up to the per-window sums (nwin XYZZ records of 128 B, about
 * 2 KiB), the ranks all-gather them, and one host combines: add the parts window by window, Horner
 * over the windows, normalise.  All ranks must use the same window layout: rank 0 (or every rank, with the same n)
 * calls porla_msm_plan and the returned *c_out is passed back as `window_bits` / `c` of the two calls below.  *c_out
 * is a plan code: bits 0..7 the window size, bit 8 set = scalars split with the GLV endomorphism (then nwin counts the
 * windows of one half), bit 9 set = not split.  A plain window size (no bit 8 / 9) lets each call decide by itself. */
#define PORLA_PLAN_WINDOW(code) ((code) & 0xff)
#define PORLA_PLAN_GLV_ON 0x100
#define PORLA_PLAN_GLV_OFF 0x200
/* Fixed-base form of the sharded MSM: every part's table carries the window expansion of porla_table_precompute with the
 * SAME window size PORLA_PLAN_WINDOW(code); all windows then share one bucket set and a part contributes ONE XYZZ sum
 * (nwin = 1 in porla_msm_finalize_host).  An SRS is a fixed base, so the expansion is built once per table. */
#define PORLA_PLAN_FIXED 0x400
void porla_msm_plan(int curve, int64_t n, int64_t nbatch, int window_bits, int* c_out, int* nwin_out);
void porla_msm_window_sums_device(const porla_table* t, const void* d_scalars, int64_t n, int scalar_fmt,
                                  int window_bits, void* d_window_sums, void* cuda_stream);
void porla_msm_finalize_host(int curve, const void* h_window_sums, int64_t nparts, int nwin, int c,
                             int out_fmt, void* out64);
/* Multi-GPU combine: parts[k*nbatch + m] (k < count) are XYZZ partials gathered from the ranks. */
void porla_msm_combine_device(int curve, const void* d_parts, int64_t count, int64_t nbatch,
                              int out_fmt, void* d_out, void* cuda_stream);
/* ---- One MSM over several GPUs of the box, inside the call (one process, one worker thread per device): the
 * reference partitions a large multi-exponentiation over 8 host threads by contiguous point range and adds the
 * partial sums (Client.hpp:747-787, Server.hpp:331-360); here the ranges go to the devices, every device runs the
 * pipeline up to its per-window sums (about 2 KiB) and the calling thread combines them.
 *   - compute_multi_exp / porla_msm_host do this by themselves for large calls when the process owns several devices:
 *     PORLA_DEVICES=k caps the fan-out (1 = off); a process pinned to one device by PORLA_DEVICE / LOCAL_RANK (one
 *     process per GPU under torchrun) stays on it unless PORLA_DEVICES says otherwise; PORLA_FANOUT_MIN = terms per
 *     device below which fewer devices are used (default 2^16).
 *   - porla_mtable: a point table resident in HBM, range-sharded over `ndev` devices (0 = all visible) at creation;
 *     an MSM over it moves only the scalars (host form) or nothing (resident form: d_scalars_per_part[p] is a device
 *     pointer ON the device of part p holding that part's scalars). */
int porla_device_count(void);
typedef struct porla_mtable porla_mtable;
porla_mtable* porla_mtable_create(int curve, const void* h_points, int64_t n, int point_fmt, int ndev);
int porla_mtable_devices(const porla_mtable* mt);
int64_t porla_mtable_len(const porla_mtable* mt);
void porla_mtable_range(const porla_mtable* mt, int part, int* device, int64_t* first, int64_t* count);
void porla_mtable_msm_host_scalars(const porla_mtable* mt, const void* h_scalars, int scalar_fmt, int out_fmt, void* out64);
void porla_mtable_msm_resident(const porla_mtable* mt, void* const* d_scalars_per_part, int scalar_fmt, int out_fmt, void* out64);
/* Copies one part's scalars (count(part) x 32 B, host) into a fresh buffer on that part's device / frees it. */
void* porla_mtable_scalars_upload(const porla_mtable* mt, int part, const void* h_scalars_of_part);
void porla_mtable_scalars_free(const porla_mtable* mt, int part, void* d_scalars);
void porla_mtable_destroy(porla_mtable* mt);
/* The fan-out of compute_multi_exp with an explicit device count (0 = all visible): host scalars and points, the
 * point range split over `ndev` devices, each copying and multiplying its range concurrently. */
void porla_msm_host_devices(int curve, const void* scalars, const void* points, int64_t n, int scalar_fmt, int point_fmt,
                            int ndev, void* out64);
/* Bytes that reached the device through the pinned-ring copy pool so far (host buffers that are not page-locked,
 * which is what the reference's callers pass: `new[]` arrays, Client.hpp:124-127). */
uint64_t porla_debug_copy_ring_bytes(void);
/* GB/s of the library's host-to-device copy path for a caller-provided host buffer (development aid). */
double porla_debug_h2d_rate(const void* h_src, uint64_t bytes, int reps);

/* Host-buffer MSM (H2D + import + MSM + D2H inside): what compute_multi_exp and the secp256k1
 * adapter are built on.  out: nbatch*64 B. */
void porla_msm_host(int curve, const void* scalars, const void* points, int64_t n, int64_t nbatch,
                    int scalar_fmt, int point_fmt, void* out);
int porla_choose_window(int curve, int64_t n, int64_t nbatch);
/* Per-stage CUDA-event timing of the most recent porla_msm_device call: ms_out[0..5] = count,
 * scan, scatter, accumulate, reduce, finalize.  Returns the number of stages (0 when disabled). */
void porla_stage_timing_enable(int on);
int porla_stage_timing_read(float* ms_out);

/* Batched single-scalar multiplication out[i] = k_i * table[i] (table of length 1: fixed base).  A length-1 table that
 * carries a look-up table (porla_table_precompute with window_bits = 0) is multiplied as a sum of nwin table entries per
 * scalar, without doublings; every other table uses double-and-add.  The output bytes are the same either way. */
void porla_scalar_mul_batch_device(const porla_table* t, const void* d_scalars, int64_t n,
                                   int scalar_fmt, int out_fmt, void* d_out, void* cuda_stream);

/* One radix-2 butterfly stage of Porla's "FFT in the exponent" (CRebuild / mix, Server.hpp:1548-1687,
 * :1209-1328; Client.hpp:921-976), which the reference issues as mult_point + add_point + neg_point +
 * add_point per butterfly (main.go:196-222): for every j < m/2 and k = j, j + m, j + 2m, ... < n
 *       t = w_j * P[k + m/2];   P[k] <- P[k] + t;   P[k + m/2] <- P[k] - t
 * `twiddles` holds the m/2 scalars w_j (32 bytes each, reduced mod the group order).  m is a power of
 * two >= 2 dividing n.  The device form works in place on a resident table (all log2 n stages of a
 * rebuild run without leaving HBM: porla_table_create, one call per stage, porla_table_export); the
 * host-buffer form does one stage on n x 64-byte gnark Marshal records in place.  Either curve. */
void porla_butterfly_stage_device(porla_table* t, int64_t m, const void* twiddles, int scalar_fmt,
                                  int twiddles_on_device, void* cuda_stream);
extern void bn254_butterfly_stage(GoSlice* points, GoInt n, GoInt m, GoSlice* twiddles);

/* The same stage on the DATA blocks (Server.hpp:1582-1588, :1240-1246; SURVEY 8(f)4): for every butterfly (k, k + m/2) and
 * every chunk p,  t = v_j * X[k + m/2][p];  X[k][p] = (u + t) % LCM;  X[k + m/2][p] = (u - t) % LCM  with u = X[k][p].
 * blocks: n_blocks x chunks chunks of 64 bytes (little-endian integers below LCM), updated in place; twiddles: m/2 values
 * of 32 bytes, little-endian (the v_j of the MAC stage, as integers); lcm_le64: LCM (utils.h:42-43, 64 bytes LE, at least
 * 2^479).  Host-buffer and device-resident forms. */
void porla_data_butterfly_stage(void* blocks, int64_t n_blocks, int64_t chunks, int64_t m, const void* twiddles_le32,
                                const void* lcm_le64);
void porla_data_butterfly_stage_device(void* d_blocks, int64_t n_blocks, int64_t chunks, int64_t m, const void* d_twiddles_le32,
                                       const void* lcm_le64, void* cuda_stream);

/* Batched Server::align_MAC, KZG branch (Server.hpp:478-562; SURVEY 8(f)2): for each of `batch` data blocks of
 * n_samples chunks A[i] -- 64-byte little-endian integers below LCM = PRIME_MODULUS * r (utils.h:37-44) --
 *       mod = A[i] % PRIME_MODULUS;   c[i] = (mod - A[i]) % r;   A[i] = mod;   align = kzg.Commit(c)
 * in ONE launch sequence (limb arithmetic and the batch of fixed-base MSMs on the GPU).  `data` is updated in
 * place (upper 32 bytes of every chunk become zero); align_out receives batch x 64 bytes, the values the
 * reference adds to the alignment MACs with bn254_add (Server.hpp:560). */
extern void bn254_align_mac_batch(GoSlice* data, GoInt batch, GoSlice* align_out);

/* Server::audit's block aggregation and its alignment, KZG branch (Server.hpp:790-828 and 903 -> 478-562; SURVEY 8(f)4):
 *       B[j] = sum_i coefs[i] * blocks[i][j]                       plain integers, no modulus (Server.hpp:798-800)
 *       mod  = B[j] % PRIME_MODULUS;  c[j] = (mod - B[j]) % r;  B[j] = mod;   align = kzg.Commit(c)
 * coefs: n x 4 bytes little-endian, the 31-bit audit coefficients (Client.hpp:700); blocks: n x n_samples chunks of
 * 64 bytes (little-endian integers below LCM, utils.h:42).  b_out receives n_samples x 32 bytes big-endian (the
 * bn254_scalar form create_proof takes, Server.hpp:388-392), align_out the 64-byte value the reference adds to the
 * combined alignment MAC (Server.hpp:560).  One aggregation kernel + one look-up-table commitment. */
extern void bn254_audit_aggregate(GoSlice* coefs, GoSlice* blocks, GoInt n, GoSlice* b_out, GoSlice* align_out);

/* ---- secp256k1 (IPA mode).  Mirrors of the reference structs (field_5x52.h:12-21,
 * group.h:13-28, scalar_4x64.h:13-15, util.h:19-22, ecmult.h:32). */
typedef struct { uint64_t n[5]; } porla_secp256k1_fe;
typedef struct { porla_secp256k1_fe x, y; int infinity; } porla_secp256k1_ge;       /* 88 B */
typedef struct { porla_secp256k1_fe x, y, z; int infinity; } porla_secp256k1_gej;   /* 128 B */
typedef struct { uint64_t d[4]; } porla_secp256k1_scalar;                           /* 32 B */
typedef struct { void (*fn)(const char* text, void* data); const void* data; } porla_secp256k1_callback;
typedef int (porla_secp256k1_ecmult_multi_callback)(porla_secp256k1_scalar* sc, porla_secp256k1_ge* pt,
                                                    size_t idx, void* data);
/* Drop-in for the static secp256k1_ecmult_multi_var (ecmult_impl.h:814-860): r = inp_g_sc*G +
 * sum_i sc_i*pt_i.  `scratch` is accepted and ignored (HBM scratch is managed internally).
 * Returns 1 on success, 0 if the callback fails; r is set to infinity first.  The result is
 * returned with z = 1 and normalised limbs. */
int porla_secp256k1_ecmult_multi_var(const porla_secp256k1_callback* error_callback, void* scratch,
                                     porla_secp256k1_gej* r, const porla_secp256k1_scalar* inp_g_sc,
                                     porla_secp256k1_ecmult_multi_callback cb, void* cbdata, size_t n);
/* Generators resident in HBM for IPA mode: Porla multiplies the same `generators[]` array in every
 * commitment, align_MAC and inner-product round (data.pt = &generators[start_chunk], Server.hpp:347,507,
 * 2345,2395; Client.hpp:393,1588).  Upload them once (any field magnitude, infinity flags honoured), then
 * r = sum_i scalars[i] * generators[first + i] with only the scalars crossing PCIe.  Same result
 * conventions as porla_secp256k1_ecmult_multi_var: r is set to infinity first, n == 0 returns 1; returns 0 if the table
 * is NULL or not secp256k1 or the range leaves it. */
porla_table* porla_secp256k1_table_create(const porla_secp256k1_ge* points, size_t n);
int porla_secp256k1_ecmult_multi_table(const porla_table* t, size_t first, const porla_secp256k1_scalar* scalars,
                                       size_t n, porla_secp256k1_gej* r);
/* Per-block commitments of an IPA-mode client or server in one call (Client::initialize's Sum A_i (alpha g_i) over 128
 * chunks, Client.hpp:377-406 / :393; Server::compute_commitment, Server.hpp:329-360 / :347):
 *       r[b] = sum_i scalars[b n + i] * t[first + i]     for b < batch
 * scalars: batch x n secp256k1_scalar, taken mod n.  One batch of look-up-table sums over the resident table, the same
 * path as porla_secp256k1_ecmult_multi_table (which is this entry with batch = 1).  With h appended to the alpha-generator
 * table and n_chunks + 1 scalars per block (the chunks, then the PRF value) each r[b] is the block's whole MAC,
 * commitment plus complement.  Results: z = 1, normalised limbs, infinity as gej_set_infinity writes it.  Returns 0 (r
 * untouched) for a NULL or non-secp256k1 table, first + n beyond the table, or n * batch >= 2^31, else 1; batch == 0 does
 * nothing and n == 0 sets every r[b] to infinity, neither touching the device.  Calls of at most 4 blocks and 4 096 terms
 * lease a staging slot of their own, so Porla's pool threads overlap on the device. */
int porla_secp256k1_ecmult_multi_table_batch(const porla_table* t, size_t first, const porla_secp256k1_scalar* scalars,
                                             size_t n, size_t batch, porla_secp256k1_gej* r);
/* The client's MAC complements batched (secp256k1_ecmult_const, ecmult_const_impl.h:137, one call per PRF value in
 * Client::initialize after CRebuild, in every update and in Client::audit's precomputation, Client.hpp:639-654):
 *       r[i] = scalars[i] * h     for i < n
 * base: a length-1 secp256k1 table holding h (porla_secp256k1_table_create(&h, 1), which also builds the look-up table of
 * its window multiples); scalars: n secp256k1_scalar as stored, not reduced (taken mod n).  k_fixed_base_mul: one thread
 * per scalar, a sum of at most 32 look-up-table entries, no doublings.  Results: z = 1, normalised limbs, infinity as
 * gej_set_infinity writes it (every r[i] when h is infinity).  Returns 0 (r untouched) for a NULL or non-secp256k1 base, a
 * base whose length is not 1, or n >= 2^31, else 1; n == 0 does not touch the device.  Calls of at most 4 scalars lease a
 * staging slot of their own.  Below 4 scalars, one porla_secp256k1_ecmult_multi_table(base, 0, &k, 1, &r) per scalar is
 * faster (profiles/r06_ipa_client_times.txt). */
int porla_secp256k1_ecmult_const_batch(const porla_table* base, const porla_secp256k1_scalar* scalars, size_t n,
                                       porla_secp256k1_gej* r);
/* Server::inner_product_prove (Server.hpp:2279-2443; SURVEY 8(f)3) over a resident table: entries 0 .. n-1 are the
 * generators (n = NUM_CHUNKS, a power of two >= 4) and entry n is the point u (Server.hpp:2376).  a, b: n scalars of 32
 * bytes, little-endian (convert_ZZ_to_arr, utils.h:353-364), any value below 2^256.  Each round's L and R are one
 * look-up-table multi-exponentiation over the whole table; the Fiat-Shamir object (one secp256k1_sha256 finalized again
 * and again, hash_impl.h:151-165), the inner products and the folding of a, b run on the host.  Writes the proof --
 * <a, b> (32 B) | per round L, R (33 B SEC1 each) | a0 b0 a1 b1 (32 B each): 32 + (log2 n - 1) * 66 + 128 bytes
 * (Server.hpp:856) -- and returns its length (0: bad arguments). */
size_t porla_secp256k1_inner_product_prove(const porla_table* gens_and_u, size_t n, const unsigned char* a_le32,
                                           const unsigned char* b_le32, unsigned char* proof);
/* Client::inner_product_verify (Client.hpp:1465-1630) over the same table (generators followed by u): returns 1 when the
 * two points the reference compares are equal, 0 otherwise (also for a malformed proof: bad SEC1 tag, x not on the
 * curve).  `commitment` is the Jacobian MAC_Block the client holds.  One variable-base multi-exponentiation over the
 * proof's L / R points and one look-up-table multi-exponentiation over the table. */
int porla_secp256k1_inner_product_verify(const porla_table* gens_and_u, size_t n, const porla_secp256k1_gej* commitment,
                                         const unsigned char* proof);
/* One stage of the FFT in the exponent on IPA-mode MACs (the rebuild butterflies of Server.hpp:1548-1830 / Client.hpp:921-976,
 * secp256k1_ecmult + 2 gej_add_var each), in place: for every j < m/2, k = j, j+m, ... < n
 *   t = w_j * P[k + m/2];  P[k] <- P[k] + t;  P[k + m/2] <- P[k] - t
 * points: n secp256k1_gej (any z, any field magnitude, infinity flag honoured); twiddles: m/2 secp256k1_scalar, taken mod n.
 * Outputs: z = 1, normalised limbs, infinity as gej_set_infinity writes it.  Returns 0 (buffer untouched) unless m is a
 * power of two >= 2 dividing n, else 1.  Stages of at most PORLA_HOST_BUTTERFLIES butterflies (default 32) run on the
 * calling host without touching the device; larger ones on the GPU (k_butterfly_quad / k_butterfly). */
int porla_secp256k1_butterfly_stage(porla_secp256k1_gej* points, size_t n, size_t m, const porla_secp256k1_scalar* twiddles);
/* Server::align_MAC, IPA branch (Server.hpp:481-518; SURVEY 8(f)2), for `batch` blocks of n_chunks chunks -- 64-byte
 * little-endian integers below LCM = PRIME_MODULUS * n (utils.h:32) -- in ONE launch sequence:
 *       mod = A[i] % PRIME_MODULUS;   c[i] = (mod - A[i]) % n;   A[i] = mod;   align_out[b] = sum_i c[i] * gens[i]
 * `data` is updated in place (upper 32 bytes of every chunk become zero).  gens: any secp256k1 table with at least
 * n_chunks entries (porla_secp256k1_table_create; entries [0, n_chunks) are used, so the prover's generators-then-u table
 * serves as it is).  Results: z = 1, normalised limbs.  Returns 0 (buffers untouched) for a bad shape -- NULL or
 * non-secp256k1 table, n_chunks 0 or longer than the table, batch * n_chunks >= 2^31 -- else 1; batch == 0 does not touch
 * the device.  Calls of a few blocks lease a staging slot of their own, so Porla's pool threads (Server.hpp:1077-1078)
 * overlap on the device. */
int porla_secp256k1_align_mac_batch(const porla_table* gens, size_t n_chunks, void* data, size_t batch,
                                    porla_secp256k1_gej* align_out);
/* Server::audit's aggregation and its alignment, IPA branch (Server.hpp:790-828 then align_MAC; SURVEY 8(f)4):
 *       B[j] = sum_i coefs[i] * blocks[i][j]     plain integers (31-bit coefs, n x n_chunks chunks of 64 bytes LE)
 *       b_out[j] = B[j] % PRIME_MODULUS;   align_out = sum_j ((B[j] % PRIME_MODULUS - B[j]) % n) * gens[j]
 * b_out_le32: n_chunks x 32 bytes little-endian (the convert_ZZ_to_arr layout porla_secp256k1_inner_product_prove reads).
 * Returns 0 (buffers untouched) for a bad table / n_chunks as above or n >= 2^24 blocks, else 1; n == 0 gives B = 0 and an
 * infinity alignment without touching the device.  One aggregation kernel and one look-up-table commitment. */
int porla_secp256k1_audit_aggregate(const porla_table* gens, size_t n_chunks, const uint32_t* coefs, const void* blocks,
                                    size_t n, unsigned char* b_out_le32, porla_secp256k1_gej* align_out);
/* r[b] = sum_i scalars[b n + i] * points[b n + i] for b < nbatch on the MACs as stored (the audit's combined_MAC /
 * combined_align, Client::audit): points are secp256k1_gej with any z and field magnitude, infinity flag honoured;
 * scalars are taken mod n.  No host inversion: each point with z != 1 costs one inversion on the device.  Results:
 * z = 1, normalised limbs, the same as porla_secp256k1_ecmult_multi_var on the same points as secp256k1_ge.  n * nbatch
 * == 0 sets every r[b] to infinity without touching the device; n * nbatch >= 2^31 returns 0, otherwise 1. */
int porla_secp256k1_ecmult_multi_gej(const porla_secp256k1_gej* points, const porla_secp256k1_scalar* scalars, size_t n,
                                     size_t nbatch, porla_secp256k1_gej* r);
/* 33-byte SEC1 compressed form of a gej/ge result (eckey_impl.h:36-52); returns 0 for infinity. */
int porla_secp256k1_gej_serialize(const porla_secp256k1_gej* a, unsigned char out33[33]);

/* Integer-multiply roofline probe: sustained 32x32->64 multiply-accumulates per second of the
 * device.  variant 0: mad.wide.u32 (IMAD.WIDE.U32); 1: mad.lo.cc/madc.hi.cc carry chains as the
 * field code issues them; 2: 32-bit mad.lo.  Runs at least min_seconds. */
double porla_measure_pint(int variant, double min_seconds);

/* Latency probe (one block on one SM): cycles and nanoseconds per operation of a dependent chain of field
 * products (mode 0; 1 / 2: two / four independent chains per thread; 3: squarings) or point operations
 * (4: XYZZ add, 5: the same with the outlined multiplier, 6: mixed add, 7: doubling), `warps` warps. */
int porla_debug_latency(int curve, int mode, int warps, int iters, double* cycles_per_op, double* ns_per_op);
/* Parity harness of the four-lane point operations (csrc/quad.cuh): out64[i] = op(A_i, B_i) over two resident tables,
 * op 0: A + B, 1: 2A, 2: 3A + B, 3: 32A (through the P + P branch), 4: (A + B) - B, 5: 2 (A + B) via scatter / gather. */
void porla_debug_quad_op(int curve, int op, const porla_table* a, const porla_table* b, int64_t n, int point_fmt, void* out64);

/* ---- test hooks (host buffers; GPU kernels underneath) */
/* out[i] = a[i] (*) b[i], the device field product on raw 8x32 LE limbs: a*b mod p for secp256k1,
 * the Montgomery product a*b*2^-256 mod p for BN254. */
void porla_debug_field_mul(int curve, const void* a, const void* b, int64_t n, void* out);
/* Same with a selectable device routine: op 0 the product, 1 the dedicated squaring a*a, 2 the fused
 * product-sum a*b + b*(a+b) (one reduction) -- the three multipliers the mixed addition uses. */
void porla_debug_field_op(int curve, int op, const void* a, const void* b, int64_t n, void* out);
/* Host-only self-check of the pairing behind verify_proof: bilinearity identities that must hold / must fail,
 * under both hard-part routines and both Miller-loop drivers.  Returns the number of failed checks. */
int porla_debug_pairing_selfcheck(int rounds);
/* out[i] = a[i] + b[i] on external 64-byte points (host-side group law, the code behind add_point). */
void porla_debug_point_add_host(int curve, const void* a, const void* b, int64_t n, int point_fmt, void* out);

#ifdef __cplusplus
}
#endif
#endif /* PORLA_MULTIEXP_H */
