// Staging of the host-buffer calls: the shared area, the slot pool and StagedCall (staging.h).
#include <cstdlib>
#include <cstring>

#include "../../include/porla_multiexp.h"
#include "staging.h"

namespace porla {

std::mutex g_io_mu;
Staging g_stage;

namespace {

// The slots outlive the calling threads (Porla builds a fresh ThreadPool inside align_MAC, Server.hpp:487).
constexpr int kStageSlots = 16;
constexpr int64_t kSlotTerms = 4096, kSlotBatch = 4;
constexpr size_t kSlotScratch = 4u << 20;
struct StagePool {
    std::mutex mu;
    Staging slots[kStageSlots];
    bool busy[kStageSlots] = {};
};
StagePool g_pool;

constexpr int64_t kHostFinalizeMaxBatch = 4;

}  // namespace

void run_and_fetch(int curve, const PointTable& tab, const uint8_t* d_scalars, int64_t n, int64_t nbatch, MsmOptions opt,
                   uint8_t* d_scratch_out, uint8_t* out, cudaStream_t st, Staging& sg) {
    const char* force_dev = getenv("PORLA_DEVICE_FINALIZE");
    if (nbatch <= kHostFinalizeMaxBatch && !(force_dev && force_dev[0] == '1')) {
        MsmPlan p = msm_plan_table(tab, (uint32_t)n, (uint32_t)nbatch, opt);
        if (p.mode == kPlanPipeline) {   // the device must use exactly the layout the host combines (window size AND split)
            opt.window_bits = p.c;
            opt.glv = p.glv;
        }
        opt.d_window_sums = d_scratch_out;
        size_t bytes = (size_t)nbatch * p.nwin * 128;
        msm_device(curve, tab, d_scalars, (uint32_t)n, (uint32_t)nbatch, opt, nullptr, nullptr, st);
        uint8_t* h = sg.pinned(bytes);
        PORLA_CUDA(cudaMemcpyAsync(h, d_scratch_out, bytes, cudaMemcpyDeviceToHost, st));
        PORLA_CUDA(cudaStreamSynchronize(st));
        for (int64_t m = 0; m < nbatch; m++) finalize_host(curve, h + (size_t)m * p.nwin * 128, p.nwin, p.c, opt.out_fmt, out + 64 * m);
        return;
    }
    msm_device(curve, tab, d_scalars, (uint32_t)n, (uint32_t)nbatch, opt, d_scratch_out, nullptr, st);
    uint8_t* h = sg.pinned((size_t)nbatch * 64);
    PORLA_CUDA(cudaMemcpyAsync(h, d_scratch_out, (size_t)nbatch * 64, cudaMemcpyDeviceToHost, st));
    PORLA_CUDA(cudaStreamSynchronize(st));
    memcpy(out, h, (size_t)nbatch * 64);
}

StagedCall::StagedCall() : s_(&g_stage), lk_(g_io_mu) { s_->init(); }

StagedCall::StagedCall(int64_t n, int64_t nbatch) {
    if (n * nbatch <= kSlotTerms && nbatch <= kSlotBatch && !getenv("PORLA_SERIAL_CALLS")) {
        std::lock_guard<std::mutex> g(g_pool.mu);
        for (int i = 0; i < kStageSlots; i++) {
            if (!g_pool.busy[i]) {
                g_pool.busy[i] = true;
                slot_ = i;
                s_ = &g_pool.slots[i];
                break;
            }
        }
    }
    if (slot_ < 0) {
        s_ = &g_stage;
        lk_ = std::unique_lock<std::mutex>(g_io_mu);
    }
    s_->init();
}

StagedCall::~StagedCall() {
    if (slot_ >= 0) {
        std::lock_guard<std::mutex> g(g_pool.mu);
        g_pool.busy[slot_] = false;
    }
}

// nbatch * nwin window sums of 128 B, which also holds the nbatch 64-byte results of the device finaliser
void StagedCall::add_result(int curve, int64_t n, int64_t nbatch) {
    const MsmPlan p = msm_plan(curve, (uint32_t)n, (uint32_t)nbatch, 0);  // general plan: an upper bound for fixed-base too
    const size_t nwin = p.nwin > 256 ? p.nwin : 256;                       // the bitwise small-MSM plan has one window per scalar bit
    out_off_ = add((size_t)nbatch * nwin * 128);
    if (slot_ >= 0) scr_off_ = add(kSlotScratch);
}

uint8_t* StagedCall::dev() { return d_ = s_->dev(layout_.size); }

MsmOptions StagedCall::msm_options(int scalar_fmt, int out_fmt, int shared_points) const {
    MsmOptions opt;
    opt.scalar_be = scalar_fmt == PORLA_SCALAR_BE32;
    opt.out_fmt = out_fmt;
    opt.shared_points = shared_points;
    if (scr_off_) {
        opt.d_scratch = d_ + scr_off_;
        opt.scratch_bytes = kSlotScratch;
    }
    return opt;
}

void StagedCall::fetch(int curve, const PointTable& tab, const uint8_t* d_scalars, int64_t n, int64_t nbatch,
                       const MsmOptions& opt, uint8_t* out) {
    run_and_fetch(curve, tab, d_scalars, n, nbatch, opt, d_ + out_off_, out, s_->stream, *s_);
}

}  // namespace porla
