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

// Host-buffer butterfly stages (bn254_butterfly_stage, porla_secp256k1_butterfly_stage): the largest stage, in butterflies,
// that runs on the calling host, and the split of a stage's nb butterflies over host threads (body(lo, hi) per thread).
int64_t host_butterfly_limit(int curve);
void for_each_butterfly_host(int64_t nb, const std::function<void(int64_t, int64_t)>& body);

// Statistics of the copy pool (test / bench hook): bytes moved through the pinned ring so far.
uint64_t h2d_ring_bytes();

}  // namespace porla
