// Pinned staging of the small per-call tables that the stream pool (csrc/stream_pool.cu) and the packed variable-length
// forward (csrc/session.cu) upload with one cudaMemcpyAsync each call.
#include <algorithm>
#include <map>
#include <mutex>
#include <utility>

#include "common.cuh"

namespace koe {

namespace {
// per (device, stream): a ring of kDepth buffers, each guarded by an event recorded after the copy that reads it, so the
// host may run kDepth calls ahead of the device before it waits
struct Staging {
  static constexpr int kDepth = 4;
  struct Ring {
    TableStaging buf[kDepth];
    int next = 0;
  };
  std::mutex mu;
  std::map<std::pair<int, void*>, Ring> rings;
};
Staging g_staging;
}  // namespace

int acquire_table_staging(void* stream, size_t ints, TableStaging** out) {
  int dev = 0;
  KOE_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(g_staging.mu);
  Staging::Ring& r = g_staging.rings[{dev, stream}];
  TableStaging& b = r.buf[r.next];
  r.next = (r.next + 1) % Staging::kDepth;
  if (b.copied == nullptr) KOE_CUDA(cudaEventCreateWithFlags(&b.copied, cudaEventDisableTiming));
  else KOE_CUDA(cudaEventSynchronize(b.copied));
  if (b.ints < ints) {
    if (b.host != nullptr) KOE_CUDA(cudaFreeHost(b.host));
    b.host = nullptr, b.ints = 0;
    const size_t want = std::max<size_t>(ints, 1024);
    KOE_CUDA(cudaHostAlloc(&b.host, want * sizeof(int32_t), cudaHostAllocDefault));
    b.ints = want;
  }
  *out = &b;
  return KOE_OK;
}

int upload_tables(TableStaging* b, int32_t* dev_tables, size_t ints, cudaStream_t stream) {
  KOE_CUDA(cudaMemcpyAsync(dev_tables, b->host, ints * sizeof(int32_t), cudaMemcpyHostToDevice, stream));
  KOE_CUDA(cudaEventRecord(b->copied, stream));
  return KOE_OK;
}

int check_capture(void* stream, const char* what) {
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  KOE_CUDA(cudaStreamIsCapturing((cudaStream_t)stream, &cap));
  if (cap != cudaStreamCaptureStatusNone)
    return fail(KOE_E_UNSUPPORTED, "%s cannot be captured into a CUDA graph: its tables change every call", what);
  return KOE_OK;
}

}  // namespace koe
