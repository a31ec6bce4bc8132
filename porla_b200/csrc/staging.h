// Host <-> device staging shared by the C-ABI entry points (abi.cu) and the in-call multi-GPU partition (multi.cu).
//
// The reference's callers hand the library ordinary heap memory (`new[]` arrays, /root/reference/porla/Client/
// Client.hpp:124-127; GoSlices over them, Utils/utils.h:277-292), i.e. PAGEABLE memory.  A cudaMemcpyAsync from
// pageable memory is staged by the driver on the calling thread at a few GB/s; h2d_copy() instead moves such buffers
// through a ring of pinned chunks filled by a small pool of copy threads (memcpy of chunk k+1 overlaps the DMA of
// chunk k), and hands pinned / registered buffers straight to the DMA engine.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <functional>
#include <mutex>

#include "msm.h"

namespace porla {

// One device buffer for inputs/outputs of host-buffer calls + streams; every object belongs to the device that was
// current when init() ran.
struct Staging {
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;   // H2D of the next part overlaps the MSM of the current one
    cudaEvent_t ev[8] = {};
    uint8_t* d_buf = nullptr;
    size_t cap = 0;
    uint8_t* h_pinned = nullptr;
    size_t h_cap = 0;
    void init() {
        if (!stream) {
            PORLA_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
            PORLA_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
            for (auto& e : ev) PORLA_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
    }
    uint8_t* dev(size_t bytes) {
        init();
        if (bytes > cap) {
            if (d_buf) {
                PORLA_CUDA(cudaStreamSynchronize(stream));
                PORLA_CUDA(cudaStreamSynchronize(copy_stream));
                PORLA_CUDA(cudaFree(d_buf));
            }
            cap = bytes + bytes / 4 + 4096;
            PORLA_CUDA(cudaMalloc(&d_buf, cap));
        }
        return d_buf;
    }
    uint8_t* pinned(size_t bytes) {
        if (bytes > h_cap) {
            if (h_pinned) PORLA_CUDA(cudaFreeHost(h_pinned));
            h_cap = bytes + 4096;
            PORLA_CUDA(cudaMallocHost(&h_pinned, h_cap));
        }
        return h_pinned;
    }
};

// true when `p` is page-locked memory the DMA engine can read directly (cudaMallocHost / cudaHostRegister)
bool host_pointer_is_pinned(const void* p);

// Asynchronous host-to-device copy of `bytes` bytes onto the CURRENT device, ordered on `stream`: kernels launched on
// `stream` afterwards see the data.  Pinned sources: one cudaMemcpyAsync.  Pageable sources above a threshold: the
// pinned-ring copy pool.  The source buffer may be reused by the caller once the call returns ONLY for pageable
// sources; for pinned sources the usual stream ordering applies (every caller in this library synchronises the
// stream before it returns to the user, which covers both).
void h2d_copy(void* d_dst, const void* h_src, size_t bytes, cudaStream_t stream);

// The staging of the default device for the large host-buffer calls (abi.cu, abi_secp.cu) and the mutex that serialises it.
extern std::mutex g_io_mu;
extern Staging g_stage;

// Regions of one staging device buffer, each 256-byte aligned: add() every region, make ONE Staging::dev(size) call (it may
// reallocate), then form the pointers from the offsets add() returned.
struct StageLayout {
    size_t size = 0;
    size_t add(size_t bytes) {
        const size_t off = size;
        size += (bytes + 255) & ~(size_t)255;
        return off;
    }
};

// Runs nbatch MSMs and brings the nbatch*64-byte results to `out`, through sg's pinned buffer.  Few MSMs: the device stops at
// the per-window sums and the serial tail (Horner + normalisation) runs on the host, which is ~15x faster than one GPU thread;
// many MSMs: the device finaliser runs them in parallel.  d_scratch_out must hold max(nbatch*64, nbatch*nwin*128) bytes.
// Returns after `st` has been synchronised.
void run_and_fetch(int curve, const PointTable& tab, const uint8_t* d_scalars, int64_t n, int64_t nbatch, MsmOptions opt,
                   uint8_t* d_scratch_out, uint8_t* out, cudaStream_t st, Staging& sg = g_stage);

// The staging of one host-buffer call.  StagedCall(n, nbatch): calls of at most 4096 terms and 4 MSMs lease one of a few
// persistent slots (device buffer, pinned buffer, stream, scratch block) and take no global lock, so Porla's pool threads
// (Server.hpp:1077-1078, Client.hpp:377-406) overlap on the device instead of queueing behind one another; larger calls,
// small ones when every slot is taken, and every call under PORLA_SERIAL_CALLS share g_stage under g_io_mu.  StagedCall():
// always the shared area.  The staging is held until the frame is destroyed, so results read from pinned() stay valid until then.
class StagedCall {
  public:
    StagedCall();
    StagedCall(int64_t n, int64_t nbatch);
    ~StagedCall();

    // Layout phase: add() returns the offset of a region; add_result() reserves what fetch() needs for nbatch MSMs of n terms
    // (and, in a slot, the scratch block that keeps the one-launch kernels off the engine's arena).  Then ONE dev() call;
    // pointers are dev() + offset.
    size_t add(size_t bytes) { return layout_.add(bytes); }
    void add_result(int curve, int64_t n, int64_t nbatch);
    uint8_t* dev();
    // Options of an MSM that fetch() runs (scalar_fmt: PORLA_SCALAR_*, out_fmt: PORLA_POINT_*), with the slot's scratch block.
    MsmOptions msm_options(int scalar_fmt, int out_fmt, int shared_points) const;
    // run_and_fetch on the frame's stream, pinned buffer and result region.
    void fetch(int curve, const PointTable& tab, const uint8_t* d_scalars, int64_t n, int64_t nbatch, const MsmOptions& opt,
               uint8_t* out);
    Staging& staging() { return *s_; }
    cudaStream_t stream() const { return s_->stream; }
    uint8_t* pinned(size_t bytes) { return s_->pinned(bytes); }

  private:
    Staging* s_ = nullptr;
    std::unique_lock<std::mutex> lk_;   // held for the shared staging area only (and makes the frame non-copyable)
    int slot_ = -1;
    StageLayout layout_;
    size_t out_off_ = 0, scr_off_ = 0;   // scr_off_ = 0: no slot scratch block (the result region precedes it)
    uint8_t* d_ = nullptr;
};

// A window [first, first + n) of a resident table: the same points, flags, endomorphism image and look-up rows.
PointTable table_window(const PointTable& t, int64_t first, int64_t n);

// Server::align_MAC on either curve (bn254_align_mac_batch, porla_secp256k1_align_mac_batch): `batch` blocks of n chunks
// of 64 bytes (LE integers below PRIME_MODULUS * order) are reduced mod PRIME_MODULUS in place in `data`, and out receives
// batch x 64 bytes (out_fmt) of sum_i c_i * gens[i], c_i = (A_i % PRIME_MODULUS - A_i) % order.  One staging area, one
// scalar kernel, one batch of MSMs over the table's first n entries; small calls lease a staging slot.
void align_mac_core(int curve, const PointTable& gens, void* data, int64_t n, int64_t batch, int out_fmt, uint8_t* out);
// Server::audit's B = sum_j coefs[j] * blocks[j] over n blocks of `chunks` chunks, then align_MAC on B: b_mod_be receives
// chunks x 32 bytes big-endian of B % PRIME_MODULUS, out64 the alignment (out_fmt).  n < 2^24.
void audit_aggregate_core(int curve, const PointTable& gens, const void* coefs, const void* blocks, int64_t n, int64_t chunks,
                          int out_fmt, uint8_t* b_mod_be, uint8_t* out64);
// nbatch secp256k1 MSMs of n terms over Jacobian points: xyz holds canonical X, Y, Z (8 LE 32-bit limbs each) of the
// n * nbatch points, inf their infinity flags, scalars n * nbatch x 8 LE 32-bit limbs; MSM m uses terms [m n, (m + 1) n).
// One device inversion per point with Z != 1 (table_import_jacobian_secp256k1); out: nbatch x 64 bytes LE64.
void msm_host_jacobian_secp256k1(const uint32_t* xyz, const uint8_t* inf, const void* scalars, int64_t n, int64_t nbatch,
                                 uint8_t* out);

// Host-buffer butterfly stages (bn254_butterfly_stage, porla_secp256k1_butterfly_stage): the largest stage, in butterflies,
// that runs on the calling host, and the split of a stage's nb butterflies over host threads (body(lo, hi) per thread).
int64_t host_butterfly_limit(int curve);
void for_each_butterfly_host(int64_t nb, const std::function<void(int64_t, int64_t)>& body);

// Statistics of the copy pool (test / bench hook): bytes moved through the pinned ring so far.
uint64_t h2d_ring_bytes();

}  // namespace porla

// The opaque handle of include/porla_multiexp.h.
struct porla_table {
    porla::PointTable t;
};

namespace porla {
// n products k_i * B over the ONE point of a length-1 table (compute_digest_complement_batch, porla_secp256k1_ecmult_const_batch):
// host scalars (n x 32 bytes, scalar_fmt) copied in, porla_scalar_mul_batch_device (k_fixed_base_mul over the table's
// look-up table); returns call's pinned buffer holding the n x 64 result bytes (out_fmt).  `call` is StagedCall(1, n).
const uint8_t* fixed_base_mul_core(StagedCall& call, const porla_table* base, const void* scalars, int64_t n, int scalar_fmt,
                                   int out_fmt);
}  // namespace porla
