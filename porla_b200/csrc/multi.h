// In-call multi-GPU partition of one MSM and the pipelined host-buffer MSM it is built from (internal to
// libmultiexp.so).  The reference partitions a large multi-exponentiation INSIDE the call: thread t of 8 takes the
// contiguous range [t*n/8, (t+1)*n/8) and the partial sums are added serially (/root/reference/porla/Client/
// Client.hpp:747-787, Server/Server.hpp:331-360).  Here the partition is over the GPUs of the box: one persistent
// worker thread per device, each with its own stream, staging buffers and engine context; every device runs the
// pipeline over its point range up to the per-window sums and the calling thread combines them.
#pragma once
#include <stdint.h>

#include <functional>

#include "msm.h"
#include "staging.h"

namespace porla {

// Number of devices a call of `n` terms fans out over: 1 below the threshold, when the process is pinned to one
// device (PORLA_DEVICE / LOCAL_RANK) or when PORLA_DEVICES=1; else min(visible devices, PORLA_DEVICES).
int fanout_devices(int64_t n);

// Runs fn(part) for part = 0 .. ndev-1 concurrently, part p on worker thread p, which drives device part_device(p)
// (= p while ndev does not exceed the visible devices) and holds a DeviceScope for it; returns when all are done.
// Calls from several user threads are serialised.
void run_on_devices(int ndev, const std::function<void(int)>& fn);
int part_device(int part);
// The staging area of the calling worker thread's device (valid inside run_on_devices only).
Staging& worker_staging();

// One MSM over host buffers on the CURRENT device, streamed in parts that accumulate into one bucket set (the copy of
// part h+1 runs under part h's kernels): writes plan.nwin window sums (128 B each) to h_ws and returns after the stream
// has been synchronised.  `plan` must be a pipeline plan; all parts of one MSM, on every device, share it.
void msm_host_pipelined(Staging& sg, int curve, const uint8_t* scalars, const uint8_t* points, int64_t n, int scalar_fmt,
                        int point_fmt, const MsmPlan& plan, uint8_t* h_ws);

// The n-term MSM over host buffers partitioned over `ndev` devices (devices 0 .. ndev-1), result to out64.
void msm_host_fanout(int curve, const uint8_t* scalars, const uint8_t* points, int64_t n, int scalar_fmt, int point_fmt,
                     int ndev, uint8_t* out64);

}  // namespace porla
