// Host-side internals shared by api_dev.cc / lr_host.cc / multi_gpu.cc / h2d.cc / the plugin ABI layer.
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <cstdint>
#include <cstddef>
#include <string>
#include <vector>
#include <deque>
#include <memory>
#include <thread>
#include <mutex>
#include <condition_variable>
#include <future>
#include <functional>
#include "../../../include/pdsb.h"

namespace pdsb {

void* pinned_alloc(size_t bytes);
void pinned_free(void* p);
int thread_streams(cudaStream_t* compute, cudaStream_t* copy);

// NVTX range per host phase (SURVEY.md §5: the reference has no tracing; nsys / ncu --nvtx group by these names)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

// null policy of the reference (src/linear/mod.rs:34-66)
enum class NullKind { RAISE, SKIP, SKIP_WINDOW, IGNORE, FILL, FILL_WINDOW };
struct NullPolicy { NullKind kind; double fill; };
// returns 0 / 1 ("Invalid NullPolicy.")
int parse_null_policy(const char* s, NullPolicy* out);

int solver_from_string(const char* s);   // lr/mod.rs:18-27
int se_type_from_string(const char* s);  // linear_regression.rs:122-132

// ---- host -> device copies (h2d.cc) ----
// One contiguous host range -> one device range.  Pinned sources go straight to the copy engine; pageable sources
// (what Polars hands a plugin) are staged through a per-device ring of pinned slots by a few host threads, so the
// page-by-page driver path (a single staging thread) is never taken for large buffers.
struct H2DSeg { void* dst; const void* src; size_t bytes; };
// Enqueue all copies; on return `s` is ordered after every one of them (the host may still be copying nothing: all
// staging memcpy()s are complete on return, only DMA may be in flight).  Destinations must have been allocated on `s`.
int h2d_execute(const std::vector<H2DSeg>& segs, cudaStream_t s);
// statistics of the last h2d_execute on this thread: bytes that took the staged (pageable) route
size_t h2d_last_staged_bytes();

// ---- multi-GPU (multi_gpu.cc) ----
struct DeviceWorker {
  int device;
  std::thread th;
  std::mutex mu;
  std::condition_variable cv;
  std::deque<std::packaged_task<int()>> q;
  bool stop = false;
  explicit DeviceWorker(int dev);
  ~DeviceWorker();
  std::future<int> submit(std::function<int()> fn);
};
struct DeviceGroup {
  std::vector<int> devices;
  std::vector<void*> comms;                            // ncclComm_t per device (in-process communicator)
  std::vector<std::unique_ptr<DeviceWorker>> workers;  // one persistent thread per device
  ~DeviceGroup();
};
DeviceGroup* active_group();                 // nullptr: single-device operation
int group_allreduce_f64(DeviceGroup* g, int idx, double* buf, size_t count, cudaStream_t s);
bool world_enabled();                        // one-process-per-GPU communicator joined (pdsb_comm_init_rank)
int world_size();
int world_rank();
int world_allreduce_f64(double* buf, size_t count, cudaStream_t s);
int world_allgather_f64(const double* send, double* recv, size_t count, cudaStream_t s);

// GLM by IRLS on a device-resident column-major X and y (glm_host.cc): beta (device, p + add_bias) receives the
// coefficients, *n_iter the number of weighted least-squares solves.  Synchronises `s` once per iteration.
int glm_irls(const double* X, int64_t ldx, const double* y, int64_t n, int p, int add_bias, int family, int64_t max_iter,
             double tol, double* beta, int64_t* n_iter, cudaStream_t s);

}  // namespace pdsb
