// Error plumbing, pinned staging ring, CUDA-graph capture (graphs.cuh), misc C-ABI entry points.
#include "common.cuh"
#include "graphs.cuh"

#include <atomic>
#include <cstdlib>
#include <cstring>

namespace gcrl {

static thread_local std::string g_last_error;

void set_last_error(const std::string &m) { g_last_error = m; }

int sm_count() {
  static int cached = 0;
  if (!cached) {
    int dev = 0, n = 0;
    GCRL_CUDA(cudaGetDevice(&dev));
    GCRL_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
    cached = n > 0 ? n : 148;
  }
  return cached;
}

bool pdl_enabled(int cls) {
  static int mask = -1;
  if (mask < 0) {
    const char *e = getenv("GCRL_NO_PDL");
    const char *m = getenv("GCRL_PDL_MASK");
    mask = (e && e[0] == '1') ? 0 : (m ? atoi(m) : (PDL_FUSED | PDL_OPTIM));
  }
  return (mask & cls) != 0;
}

static std::atomic<uint64_t> g_launches{0};
void count_launch(uint64_t n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
uint64_t launch_counter() { return g_launches.load(std::memory_order_relaxed); }

void PinnedRing::init(size_t bytes) {
  slot_bytes = (bytes + 255) & ~size_t(255);
  GCRL_CUDA(cudaMallocHost(&base, slot_bytes * kSlots));
  for (int i = 0; i < kSlots; ++i) {
    GCRL_CUDA(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
    used[i] = false;
  }
  next = 0;
}

void PinnedRing::destroy() {
  if (!base) return;
  for (int i = 0; i < kSlots; ++i) cudaEventDestroy(ev[i]);
  cudaFreeHost(base);
  base = nullptr;
}

char *PinnedRing::acquire(size_t bytes, int *slot) {
  if (bytes > slot_bytes) {
    // grow: drain everything in flight, then reallocate
    for (int i = 0; i < kSlots; ++i)
      if (used[i]) { GCRL_CUDA(cudaEventSynchronize(ev[i])); used[i] = false; }
    GCRL_CUDA(cudaFreeHost(base));
    base = nullptr;
    slot_bytes = (bytes * 2 + 255) & ~size_t(255);
    GCRL_CUDA(cudaMallocHost(&base, slot_bytes * kSlots));
  }
  int s = next;
  next = (next + 1) % kSlots;
  if (used[s]) { GCRL_CUDA(cudaEventSynchronize(ev[s])); used[s] = false; }
  *slot = s;
  return base + size_t(s) * slot_bytes;
}

void PinnedRing::release(int slot, cudaStream_t st) {
  GCRL_CUDA(cudaEventRecord(ev[slot], st));
  used[slot] = true;
}

bool graphs_enabled() {
  const char *ng = getenv("GCRL_B200_NO_GRAPH");
  return !(ng && ng[0] == '1');
}

void begin_capture(cudaStream_t cap) { GCRL_CUDA(cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal)); }

GraphRec end_capture(cudaStream_t cap, uint64_t kernels) {
  cudaGraph_t graph = nullptr;
  GCRL_CUDA(cudaStreamEndCapture(cap, &graph));
  count_launch(uint64_t(0) - kernels);
  cudaGraphExec_t exec = nullptr;
  const cudaError_t e = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  GCRL_CUDA(e);
  return GraphRec{exec, kernels};
}

void abort_capture(cudaStream_t cap) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(cap, &cs);
  if (cs == cudaStreamCaptureStatusNone) return;
  cudaGraph_t graph = nullptr;
  cudaStreamEndCapture(cap, &graph);
  if (graph) cudaGraphDestroy(graph);
}

GraphRec capture_graph(cudaStream_t cap, const std::function<void(cudaStream_t)> &body) {
  const uint64_t before = launch_counter();
  begin_capture(cap);
  try {
    body(cap);
  } catch (...) {
    abort_capture(cap);
    throw;
  }
  return end_capture(cap, launch_counter() - before);
}

void launch_graph(const GraphRec &g, cudaStream_t st) {
  GCRL_CUDA(cudaGraphLaunch(g.exec, st));
  count_launch(g.kernels);
}

}  // namespace gcrl

extern "C" {

int gcrl_abi_version(void) { return GCRL_ABI_VERSION; }

const char *gcrl_last_error(void) { return gcrl::g_last_error.c_str(); }

uint64_t gcrl_kernel_launches(void) { return gcrl::launch_counter(); }

int gcrl_device_count(int *count) {
  GCRL_API_BEGIN
  GCRL_REQUIRE(count != nullptr, "count is NULL");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    cudaGetLastError();
    n = 0;
  }
  *count = n;
  GCRL_API_END
}

}  // extern "C"
